// First-layer kernel: 3x3 stride-1 'same' convolution over a C_in <= 3 fp32 NCHW image, fused with
// batchnorm + bias + leaky-ReLU AND the 2x2/2 maxpool that follows it in every north-star cfg.
//
// Replaces, for layers 0 and 1 of yolo-voc / tiny-yolo-voc / yolo9000 / darknet19:
//   cuda_make_array(input) + fill + im2col_ongpu + gemm_ongpu + normalize + scale_bias + add_bias +
//   activate_array (convolutional_kernels.cu:77-131) + forward_maxpool_layer_kernel
//   (maxpool_layer_kernels.cu:10-48)
// by one persistent launch that reads the caller's fp32 planar image once and writes only the
// pooled bf16 padded-NHWC tensor.  The layer is HBM-bound (K = 27): per image it must move
// 3*H*W*4 bytes in and (H/2)*(W/2)*32*2 bytes out; the full-resolution activation never exists.
//
// How the im2col disappears.  A patch of (R+2) input rows x P positions is converted once to bf16
// and stored in shared memory with ONE 16-byte row per position q of a patch row:
//       row q = [ pixel q: c0 c1 c2 0 | pixel q+1: c0 c1 c2 0 ]          (8 bf16)
// In the no-swizzle K-major UMMA layout the two 16-byte K-chunks of an operand row may sit at any
// byte distance (the descriptor's leading-dimension offset); with that distance set to 32 bytes the
// second chunk of row q IS row q+2, so a K = 16 operand row reads pixels q..q+3: the three
// horizontal taps of a 3x3 filter row (+ one pixel against zero weights) in a single tcgen05.mma.
// The vertical taps are three descriptors whose start address differs by one patch row.  One
// image row of 128 positions therefore costs 3 MMAs (M = 128, N = 32, K = 16) and no data is ever
// replicated per tap.  Two accumulators hold image rows y and y+1 in the same TMEM lanes, so the
// 2x2 pool is a vertical max inside a thread and one shuffle with the neighbouring lane.
//
// Warp roles (768 threads): 0-5 converters (fp32 -> bf16 patch rows), 6 MMA issuer (+ TMEM alloc),
// 7 TMA loader (the raw fp32 box of the next patch, zero-filled outside the image by the TMA unit),
// 8-23 epilogue: four groups of four warps = (slot parity) x (channel half); the epilogue is a long
// dependent chain per thread, so it is spread over many warps, each draining 16 of the 32 channels
// of its slots (TMEM lane quarter = warp & 3).  Images whose row pitch is not a multiple of 16 bytes cannot be described by a tensor
// map; for those the converters read global memory directly.
//
// max before the affine map is exact: the host makes every alpha_f >= 0 (a filter with negative
// alpha has its weights and alpha negated, which leaves alpha*acc bit-identical), and
// x -> leaky(fma(alpha, x, beta)) is then non-decreasing in fp32, so it commutes with max.
#include "conv_plan.cuh"

#include <string.h>

namespace y2 {

constexpr int kStemProducerWarps = 6;
constexpr int kStemEpilogueWarps = 16;
constexpr int kStemThreads = (kStemProducerWarps + 2 + kStemEpilogueWarps) * 32;  // 768
constexpr int kStemN = 32;          // filters (padded)
constexpr int kStemK = 32;          // K stride of the weight matrix handed in by the host (27 used)
constexpr int kStemRows = 16;       // image rows per patch (8 pooled rows)
constexpr int kStemMaxP = 128;      // positions per patch row (tile width + 2)
constexpr int kStemStages = 2;
constexpr int kStemSlots = 4;       // TMEM slots of four 32-column accumulators (two row pairs) each
constexpr int kStemBoxW = 132;      // floats per raw row: tile width + 8, at most
constexpr int kPatchBytes = ((kStemRows + 2) * kStemMaxP + 136) * 16;  // + tail read by the junk lanes
constexpr uint32_t kStemIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kStemN >> 3) << 17) |
                                ((uint32_t)(128 >> 4) << 24);

struct StemParams {
    const float *in;   // fp32 [B][c][h][w]
    int batch, c, h, w;
    int oh, ow;        // pooled extent
    int wt;            // image columns per tile (even), P = wt + 2
    int tiles_x, tiles_y, total_tiles;
    const __nv_bfloat16 *wgt;  // [32][32], K index c*9 + r*3 + s
    const float *alpha, *beta;
    int act;
    __nv_bfloat16 *out;  // padded NHWC [B][oh+1][ow+1][out_cs]
    int out_cs;
    int use_tma;       // 1: raw fp32 planar boxes arrive through tm_in, 2: raw uint8 HWC boxes (the image is
                       // [B][H][W][3] bytes, value = byte / 255), 0: the converters load global fp32 directly
    int boxw;          // floats (mode 1) or bytes (mode 2) per raw row of the box
};

struct StemSmem {
    alignas(128) uint8_t patch[kStemStages][kPatchBytes];
    struct alignas(128) Raw { float v[3 * (kStemRows + 2) * kStemBoxW]; } raw[kStemStages];  // TMA destinations
    alignas(128) uint8_t w[3][1024];  // per filter row dr: [k-chunk 2][n 32][8 bf16]
    float alpha[kStemN], beta[kStemN];
    float lut[256];    // byte -> (float)(byte / 255.), the conversion of yolo_v2_class.cpp:141 / image.c
    alignas(8) uint64_t p_full[kStemStages], p_empty[kStemStages], r_full[kStemStages], r_empty[kStemStages];
    uint64_t t_full[kStemSlots], t_empty[kStemSlots];
    uint32_t tmem_slot;
};

// no-swizzle K-major descriptor: rows 16 B apart, 8-row groups `sbo` bytes apart, the second
// 16-byte K chunk `lbo` bytes after the first
__device__ __forceinline__ uint64_t stem_desc(uint32_t addr, uint32_t lbo, uint32_t sbo)
{
    uint64_t d = 0;
    d |= (uint64_t)((addr & 0x3FFFF) >> 4);
    d |= (uint64_t)(lbo >> 4) << 16;
    d |= (uint64_t)(sbo >> 4) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}

__device__ __forceinline__ uint2 stem_load_pixel(const StemParams &p, const float *img, int gy, int gx)
{
    float v0 = 0.f, v1 = 0.f, v2 = 0.f;
    if (gy >= 0 && gy < p.h && gx >= 0 && gx < p.w) {
        const float *s = img + (size_t)gy * p.w + gx;
        const size_t plane = (size_t)p.h * p.w;
        v0 = __ldg(s);
        if (p.c > 1) v1 = __ldg(s + plane);
        if (p.c > 2) v2 = __ldg(s + 2 * plane);
    }
    return make_uint2(pack_bf16x2(v0, v1), pack_bf16x2(v2, 0.f));
}

__device__ __forceinline__ void tma_load_3d(const void *desc, uint64_t *bar, void *smem_dst, int c0, int c1, int c2)
{
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(smem_dst)),
        "l"(desc), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

__global__ void __launch_bounds__(kStemThreads, 1)
stem_conv_pool_kernel(const __grid_constant__ CUtensorMap tm_in, const StemParams p)
{
    extern __shared__ uint8_t stem_raw[];
    StemSmem &sm = *reinterpret_cast<StemSmem *>(stem_raw + ((128u - (smem_u32(stem_raw) & 127u)) & 127u));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int P = p.wt + 2;
    const int pairs = kStemRows / 2;

    if (threadIdx.x == 0) {
        for (int i = 0; i < kStemStages; ++i) {
            mbar_init(&sm.p_full[i], kStemProducerWarps * 32);
            mbar_init(&sm.p_empty[i], 1);
            mbar_init(&sm.r_full[i], 1);
            mbar_init(&sm.r_empty[i], kStemProducerWarps * 32);
        }
        for (int i = 0; i < kStemSlots; ++i) {
            mbar_init(&sm.t_full[i], 1);
            mbar_init(&sm.t_empty[i], 256);  // both channel-half groups
        }
        fence_barrier_init();
    }
    if (warp == kStemProducerWarps) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sm.tmem_slot)),
                     "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // weights: B_dr[n][k = 4*j + c] = w[n][c*9 + dr*3 + j]  (j < 3 horizontal tap, c < C_in), else 0
    for (int e = threadIdx.x; e < 3 * kStemN * 16; e += kStemThreads) {
        const int dr = e / (kStemN * 16);
        const int n = (e / 16) % kStemN;
        const int k = e % 16;
        const int j = k >> 2, c = k & 3;
        __nv_bfloat16 v = __float2bfloat16_rn(0.f);
        if (j < 3 && c < p.c) v = p.wgt[n * kStemK + c * 9 + dr * 3 + j];
        const int off = (k >> 3) * 512 + (n >> 3) * 128 + (n & 7) * 16 + (k & 7) * 2;
        *reinterpret_cast<__nv_bfloat16 *>(sm.w[dr] + off) = v;
    }
    // the tail behind the last patch row is only ever read by discarded lanes, but must stay finite
    for (int e = threadIdx.x; e < kStemStages * kPatchBytes / 16; e += kStemThreads)
        reinterpret_cast<uint4 *>(sm.patch[0])[e] = make_uint4(0u, 0u, 0u, 0u);
    if (threadIdx.x < kStemN) {
        sm.alpha[threadIdx.x] = p.alpha[threadIdx.x];
        sm.beta[threadIdx.x] = p.beta[threadIdx.x];
    }
    if (threadIdx.x < 256) sm.lut[threadIdx.x] = (float)((double)threadIdx.x / 255.);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = sm.tmem_slot;
    const int per_img = p.tiles_x * p.tiles_y;

    if (warp < kStemProducerWarps) {
        // ===================== converters: fp32 -> bf16 patch rows =====================
        const int n_pos = (kStemRows + 2) * P;
        const uint32_t inv_p = (uint32_t)(((1u << 20) + P - 1) / P);  // e / P == (e * inv_p) >> 20 for e < 2304
        int it = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
            const int s = it % kStemStages;
            const uint32_t ph = (uint32_t)(it / kStemStages) & 1u;
            uint4 *dst = reinterpret_cast<uint4 *>(sm.patch[s]);
            if (p.use_tma == 2) {
                mbar_wait_relaxed(&sm.r_full[s], ph, 9);
                mbar_wait_relaxed(&sm.p_empty[s], ph ^ 1, 10);
                const int t = tile % per_img;
                const int tx = t % p.tiles_x;
                const int x3 = (tx * p.wt - 1) * 3;
                const uint8_t *raw = reinterpret_cast<const uint8_t *>(sm.raw[s].v) + (x3 - (x3 & ~15));
#pragma unroll 4
                for (int e = threadIdx.x; e < n_pos; e += kStemProducerWarps * 32) {
                    const int r = (int)(((uint32_t)e * inv_p) >> 20), q = e - r * P;
                    const uint8_t *px = raw + r * p.boxw + 3 * q;  // pixel q and its right neighbour, RGB bytes
                    dst[e] = make_uint4(pack_bf16x2(sm.lut[px[0]], sm.lut[px[1]]), pack_bf16x2(sm.lut[px[2]], 0.f),
                                        pack_bf16x2(sm.lut[px[3]], sm.lut[px[4]]), pack_bf16x2(sm.lut[px[5]], 0.f));
                }
                fence_proxy_async();
                mbar_arrive(&sm.p_full[s]);
                mbar_arrive(&sm.r_empty[s]);
                continue;
            }
            if (p.use_tma) {
                mbar_wait_relaxed(&sm.r_full[s], ph, 9);
                mbar_wait_relaxed(&sm.p_empty[s], ph ^ 1, 10);
                const float *raw = sm.raw[s].v;
                const int plane = (kStemRows + 2) * p.boxw;
#pragma unroll 4
                for (int e = threadIdx.x; e < n_pos; e += kStemProducerWarps * 32) {
                    const int r = (int)(((uint32_t)e * inv_p) >> 20), q = e - r * P;
                    const float *px = raw + r * p.boxw + q + 3;  // the box starts at image column x0 - 4
                    float a0 = px[0], b0 = px[1], a1 = 0.f, b1 = 0.f, a2 = 0.f, b2 = 0.f;
                    if (p.c > 1) { a1 = px[plane]; b1 = px[plane + 1]; }
                    if (p.c > 2) { a2 = px[2 * plane]; b2 = px[2 * plane + 1]; }
                    dst[e] = make_uint4(pack_bf16x2(a0, a1), pack_bf16x2(a2, 0.f), pack_bf16x2(b0, b1),
                                        pack_bf16x2(b2, 0.f));
                }
                fence_proxy_async();
                mbar_arrive(&sm.p_full[s]);
                mbar_arrive(&sm.r_empty[s]);
                continue;
            }
            const int b = tile / per_img;
            const int t = tile - b * per_img;
            const int ty = t / p.tiles_x, tx = t - ty * p.tiles_x;
            const int y0 = ty * kStemRows - 1, x0 = tx * p.wt - 1;
            const float *img = p.in + (size_t)b * p.c * p.h * p.w;
            mbar_wait_relaxed(&sm.p_empty[s], ph ^ 1, 10);
            // a warp covers 31 positions per step; lane 31 only supplies the right neighbour of lane 30 (the
            // next step recomputes it as lane 0).  Eight steps are loaded before any is consumed so that
            // 24 independent global loads per thread are in flight (one memory round trip per patch).
            constexpr int kBatch = 8;
            for (int e0 = warp * 31; e0 < n_pos; e0 += kBatch * kStemProducerWarps * 31) {
                uint2 a[kBatch];
#pragma unroll
                for (int u = 0; u < kBatch; ++u) {
                    const int e = e0 + u * kStemProducerWarps * 31 + lane;
                    const int r = e / P, q = e - r * P;
                    a[u] = stem_load_pixel(p, img, y0 + r, x0 + q);
                }
#pragma unroll
                for (int u = 0; u < kBatch; ++u) {
                    const int e = e0 + u * kStemProducerWarps * 31 + lane;
                    // a row wrap only feeds lanes that are discarded
                    const uint32_t nx = __shfl_down_sync(0xffffffffu, a[u].x, 1);
                    const uint32_t ny = __shfl_down_sync(0xffffffffu, a[u].y, 1);
                    if (lane < 31 && e < n_pos) dst[e] = make_uint4(a[u].x, a[u].y, nx, ny);
                }
            }
            fence_proxy_async();
            mbar_arrive(&sm.p_full[s]);
        }
    } else if (warp == kStemProducerWarps + 1) {
        // ===================== TMA loader: raw fp32 box of every patch =====================
        if (p.use_tma) {
            int it = 0;
            const uint32_t box_bytes = p.use_tma == 2 ? (uint32_t)((kStemRows + 2) * p.boxw)
                                                      : (uint32_t)(p.c * (kStemRows + 2) * p.boxw * 4);
            for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
                const int s = it % kStemStages;
                const uint32_t ph = (uint32_t)(it / kStemStages) & 1u;
                const int b = tile / per_img;
                const int t = tile - b * per_img;
                const int ty = t / p.tiles_x, tx = t - ty * p.tiles_x;
                mbar_wait_relaxed(&sm.r_empty[s], ph ^ 1, 8);
                if (elect_one_sync()) {
                    mbar_expect_tx(&sm.r_full[s], box_bytes);
                    // the innermost box coordinate must be 16-byte aligned: start four columns left of the tile
                    if (p.use_tma == 2)  // byte column of pixel x0 - 1, rounded down to 16 bytes
                        tma_load_3d(&tm_in, &sm.r_full[s], sm.raw[s].v, (((tx * p.wt - 1) * 3) & ~15) >> 2,
                                    ty * kStemRows - 1, b);  // the tensor map counts 32-bit words
                    else
                        tma_load_3d(&tm_in, &sm.r_full[s], sm.raw[s].v, tx * p.wt - 4, ty * kStemRows - 1, b * p.c);
                }
                __syncwarp();
            }
        }
    } else if (warp == kStemProducerWarps) {
        // ===================== MMA issuer =====================
        const uint32_t w_lo = (smem_u32(sm.w[0]) & 0x3FFFFu) >> 4;
        // descriptor words: hi = SBO 128 B | version 1; lo = address >> 4 | LBO >> 4 at bit 16
        constexpr uint32_t kHi = (128u >> 4) | (1u << 14);
        constexpr uint32_t kLboA = (32u >> 4) << 16, kLboB = (512u >> 4) << 16;
        int it = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
            const int s = it % kStemStages;
            const uint32_t ph = (uint32_t)(it / kStemStages) & 1u;
            mbar_wait(&sm.p_full[s], ph, 11);
            tc_fence_after();
            const uint32_t patch_lo = (smem_u32(sm.patch[s]) & 0x3FFFFu) >> 4;
#pragma unroll 1
            for (int h = 0; h < kStemSlots; ++h) {  // slot h: image rows 4h .. 4h+3 (two row pairs)
                mbar_wait(&sm.t_empty[h], (uint32_t)(it & 1) ^ 1, 12);
                tc_fence_after();
                if (elect_one_sync()) {
                    const uint32_t row_lo = patch_lo + (uint32_t)(4 * h * P);
#pragma unroll
                    for (int i = 0; i < 4; ++i) {  // image row 4h + i -> accumulator i of the slot
                        const uint32_t d = tmem_base + (uint32_t)(h * 128 + i * 32);
#pragma unroll
                        for (int dr = 0; dr < 3; ++dr) {
                            // patch row 4h + i + dr; the filter's three horizontal taps ride in K
                            const uint64_t adesc = ((uint64_t)kHi << 32) | (uint64_t)((row_lo + (uint32_t)((i + dr) * P)) | kLboA);
                            const uint64_t bdesc = ((uint64_t)kHi << 32) | (uint64_t)((w_lo + (uint32_t)(dr * 64)) | kLboB);
                            umma_bf16(d, adesc, bdesc, kStemIdesc, (uint32_t)(dr != 0));
                        }
                    }
                    umma_commit(&sm.t_full[h]);
                    if (h == kStemSlots - 1) umma_commit(&sm.p_empty[s]);
                }
                __syncwarp();
            }
        }
    } else {
        // ===================== epilogue: 2x2 max, affine, leaky, store =====================
        const int ew = warp - (kStemProducerWarps + 2);  // 0..15
        const int sgroup = ew >> 3;                      // slots alternate between the two slot groups
        const int chalf = (ew >> 2) & 1;                 // channels [16 chalf, 16 chalf + 16)
        const int quarter = warp & 3;
        const int m = quarter * 32 + lane;               // TMEM lane == position inside the tile row
        const int hsel = lane & 1;                       // even lane finishes 8 channels, odd lane the other 8
        const int cbase = chalf * 16 + hsel * 8;         // first channel this thread stores
        float al[8], be[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            al[q] = sm.alpha[cbase + q];
            be[q] = sm.beta[cbase + q];
        }
        int it = 0;
        // (image, tile row, tile column) advance by a constant stride: carry-propagate instead of dividing
        // per tile (two runtime divisions were 9 % of this issue-bound kernel's instructions)
        int b = (int)blockIdx.x / per_img;
        int ty = ((int)blockIdx.x - b * per_img) / p.tiles_x;
        int tx = (int)blockIdx.x - b * per_img - ty * p.tiles_x;
        const int db = (int)gridDim.x / per_img;
        const int dty = ((int)gridDim.x - db * per_img) / p.tiles_x;
        const int dtx = (int)gridDim.x - db * per_img - dty * p.tiles_x;
        const size_t row_elems = (size_t)(p.ow + 1) * p.out_cs;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
            if (it) {
                tx += dtx;
                if (tx >= p.tiles_x) { tx -= p.tiles_x; ++ty; }
                ty += dty;
                if (ty >= p.tiles_y) { ty -= p.tiles_y; ++b; }
                b += db;
            }
            const int ox = (tx * p.wt + m) >> 1;
            __nv_bfloat16 *obase = p.out + ((size_t)b * (p.oh + 1) + (size_t)ty * (kStemRows / 2)) * row_elems +
                                   (size_t)ox * p.out_cs + cbase;
            const bool col_ok = m < p.wt && ox < p.ow;
            for (int jp = 2 * sgroup; jp < pairs; jp += 4)
            for (int j = jp; j < jp + 2; ++j) {
                const int slot = j >> 1;
                if ((j & 1) == 0) {
                    mbar_wait_relaxed(&sm.t_full[slot], (uint32_t)(it & 1), 13);
                    tc_fence_after();
                }
                const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) +
                                       (uint32_t)(slot * 128 + (j & 1) * 64 + chalf * 16);
                uint32_t v[16], u[16];
                tmem_ld16(taddr, v);
                tmem_ld16(taddr + 32u, u);
                tmem_ld_wait();
                if (j & 1) {  // both row pairs of the slot are in registers
                    tc_fence_before();
                    mbar_arrive(&sm.t_empty[slot]);
                }
                // vertical max in-thread, then trade halves with the horizontal neighbour
                float mx[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const float lo = fmaxf(__uint_as_float(v[q]), __uint_as_float(u[q]));
                    const float hi = fmaxf(__uint_as_float(v[q + 8]), __uint_as_float(u[q + 8]));
                    const float send = hsel ? lo : hi;  // what the partner keeps
                    const float keep = hsel ? hi : lo;
                    const float got = __shfl_xor_sync(0xffffffffu, send, 1);
                    mx[q] = fmaxf(keep, got);
                }
                const int oy = ty * (kStemRows / 2) + j;
                if (col_ok && oy < p.oh) {
                    uint32_t pk[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        float y0 = fmaf(mx[2 * q], al[2 * q], be[2 * q]);
                        float y1 = fmaf(mx[2 * q + 1], al[2 * q + 1], be[2 * q + 1]);
                        if (p.act == Y2_ACT_LEAKY) {
                            y0 = fmaxf(y0, 0.1f * y0);
                            y1 = fmaxf(y1, 0.1f * y1);
                        }
                        pk[q] = pack_bf16x2(y0, y1);
                    }
                    *reinterpret_cast<uint4 *>(obase + (size_t)j * row_elems) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == kStemProducerWarps) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

} // namespace y2

using namespace y2;

// raise the dynamic shared-memory limit (plan time, outside any graph capture)
extern "C" int y2_stem_prepare(void)
{
    static bool attr_done[64] = {false};
    int dev = 0;
    Y2_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && !attr_done[dev]) {
        Y2_CUDA_CHECK(cudaFuncSetAttribute(stem_conv_pool_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)(sizeof(StemSmem) + 128)));
        attr_done[dev] = true;
    }
    return Y2_OK;
}

// column tile of the first-layer kernel: equal tiles of at most 124 image columns, a multiple of 4 wide
static int stem_tile_cols(int w)
{
    const int ow = w / 2;
    const int wmax = kStemMaxP - 4;
    const int nx = (2 * ow + wmax - 1) / wmax;
    int wt_cols = (2 * ow + nx - 1) / nx;
    return (wt_cols + 3) / 4 * 4;
}

static int stem_u8_boxw(int w) { return ((stem_tile_cols(w) + 3) * 3 + 15 + 15) / 16 * 16; }

// the image sizes y2_stem_conv_pool_u8 accepts (callers fall back to the resize / float path otherwise)
extern "C" int y2_stem_u8_supported(int h, int w)
{
    if (h < 2 || w < 2) return 0;
    const int boxw = stem_u8_boxw(w);
    return (3 * w) % 16 == 0 && boxw <= 3 * w && kStemRows + 2 <= h &&
           (size_t)(kStemRows + 2) * boxw <= sizeof(StemSmem::Raw);
}

// in: fp32 planar [B][c][h][w] when !u8, uint8 interleaved [B][h][w][3] when u8
static int stem_launch(const void *in, bool u8, int batch, int c, int h, int w, const void *wt, int npad,
                       const float *alpha, const float *beta, int act, void *out, int out_cs, y2_stream_t s)
{
    if (!in || !wt || !alpha || !beta || !out || batch <= 0 || c <= 0 || c > 3 || h < 2 || w < 2 || npad != kStemN ||
        out_cs % 8 || out_cs < kStemN || ((uintptr_t)out & 15) || ((uintptr_t)wt & 15) ||
        (act != Y2_ACT_LEAKY && act != Y2_ACT_LINEAR)) {
        set_error("y2_stem_conv_pool: invalid arguments (c=%d h=%d w=%d npad=%d out_cs=%d act=%d)", c, h, w, npad,
                  out_cs, act);
        return Y2_EINVAL;
    }
    StemParams p;
    p.in = u8 ? nullptr : (const float *)in;
    p.batch = batch;
    p.c = c;
    p.h = h;
    p.w = w;
    p.oh = h / 2;
    p.ow = w / 2;
    // equal column tiles of at most 124 image columns, a multiple of 4 wide (16-byte aligned TMA boxes)
    const int wt_cols = stem_tile_cols(w);
    p.wt = wt_cols;
    p.tiles_x = (2 * p.ow + wt_cols - 1) / wt_cols;
    p.tiles_y = (p.oh + kStemRows / 2 - 1) / (kStemRows / 2);
    const long long total = (long long)batch * p.tiles_x * p.tiles_y;
    if (total > 0x7fffffffLL) return Y2_EINVAL;
    p.total_tiles = (int)total;
    p.wgt = (const __nv_bfloat16 *)wt;
    p.alpha = alpha;
    p.beta = beta;
    p.act = act;
    p.out = (__nv_bfloat16 *)out;
    p.out_cs = out_cs;
    const size_t smem = sizeof(StemSmem) + 128;
    int rc = y2_stem_prepare();
    if (rc != Y2_OK) return rc;
    // raw boxes through TMA when the image rows are 16-byte aligned; the tensor map is encoded per call
    // (the input pointer is the caller's) and travels by value in the launch / graph node
    CUtensorMap tm;
    memset(&tm, 0, sizeof(tm));
    p.use_tma = 0;
    EncodeTiledFn enc = get_encode_fn();
    if (u8) {
        // bytes (x0 - 1)*3 .. (x0 + wt + 2)*3 of a row, from the 16-byte boundary below the first one
        p.boxw = stem_u8_boxw(w);
        if (!enc || c != 3 || ((uintptr_t)in & 15) || !y2_stem_u8_supported(h, w)) {
            set_error("y2_stem_conv_pool_u8: needs 3 channels, a width that is a multiple of 16 and at least %d rows "
                      "(h=%d w=%d c=%d)", kStemRows + 2, h, w, c);
            return Y2_EINVAL;
        }
        // described as 32-bit words: a box dimension is limited to 256 elements, a row of bytes would not fit
        cuuint64_t gdim[3] = {(cuuint64_t)w * 3 / 4, (cuuint64_t)h, (cuuint64_t)batch};
        cuuint64_t gstr[2] = {(cuuint64_t)w * 3, (cuuint64_t)w * h * 3};
        cuuint32_t box[3] = {(cuuint32_t)p.boxw / 4, (cuuint32_t)(kStemRows + 2), 1u};
        cuuint32_t estr[3] = {1, 1, 1};
        CUresult r = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, const_cast<void *>(in), gdim, gstr, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            set_error("y2_stem_conv_pool_u8: cuTensorMapEncodeTiled failed: CUresult %d", (int)r);
            return Y2_ECUDA;
        }
        p.use_tma = 2;
    } else {
        p.boxw = p.wt + 8;  // image columns x0 - 4 .. x0 + wt + 3
        // a box never exceeds the tensor it slides over
        if (enc && w % 4 == 0 && ((uintptr_t)in & 15) == 0 && p.boxw <= kStemBoxW && p.boxw <= w && kStemRows + 2 <= h) {
            cuuint64_t gdim[3] = {(cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)batch * c};
            cuuint64_t gstr[2] = {(cuuint64_t)w * 4, (cuuint64_t)w * h * 4};
            cuuint32_t box[3] = {(cuuint32_t)p.boxw, (cuuint32_t)(kStemRows + 2), (cuuint32_t)c};
            cuuint32_t estr[3] = {1, 1, 1};
            CUresult r = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void *>(in), gdim, gstr, box, estr,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            p.use_tma = (r == CUDA_SUCCESS);
        }
    }
    const int sms = sm_count();
    const int grid = p.total_tiles < sms ? p.total_tiles : sms;
    stem_conv_pool_kernel<<<grid, kStemThreads, smem, to_stream(s)>>>(tm, p);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_stem_conv_pool(const float *in, int batch, int c, int h, int w, const void *wt, int npad,
                                 const float *alpha, const float *beta, int act, void *out, int out_cs,
                                 y2_stream_t s)
{
    return stem_launch(in, false, batch, c, h, w, wt, npad, alpha, beta, act, out, out_cs, s);
}

extern "C" int y2_stem_conv_pool_u8(const unsigned char *in_hwc, int batch, int h, int w, const void *wt, int npad,
                                    const float *alpha, const float *beta, int act, void *out, int out_cs,
                                    y2_stream_t s)
{
    return stem_launch(in_hwc, true, batch, 3, h, w, wt, npad, alpha, beta, act, out, out_cs, s);
}
