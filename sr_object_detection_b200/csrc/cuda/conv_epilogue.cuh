// Shared epilogue piece of the slab / pair convolution kernels.
#pragma once
#include "conv_plan.cuh"

namespace y2 {

// one 32-column chunk of one accumulator row: affine + activation + store
template <int ACT>
__device__ __forceinline__ void slab_epilogue_chunk(const SlabParams &prm, const uint32_t (&v)[32], const float2 *sab,
                                                    int c0, int n0, int p, int b, int y, int x, bool in_range,
                                                    bool valid)
{
    float f[32];
    const float4 *ab4 = reinterpret_cast<const float4 *>(sab + c0);
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const float4 q = ab4[j];  // (alpha, beta) of two filters
        float t0 = fmaf(__uint_as_float(v[2 * j]), q.x, q.y);
        float t1 = fmaf(__uint_as_float(v[2 * j + 1]), q.z, q.w);
        if (ACT == Y2_ACT_LEAKY) {  // max(t, 0.1 t) == (t > 0 ? t : 0.1 t) for every finite t
            t0 = fmaxf(t0, 0.1f * t0);
            t1 = fmaxf(t1, 0.1f * t1);
        } else if (ACT == Y2_ACT_LOGISTIC) {
            t0 = 1.f / (1.f + __expf(-t0));
            t1 = 1.f / (1.f + __expf(-t1));
        }
        f[2 * j] = t0;
        f[2 * j + 1] = t1;
    }
    const int ch0 = n0 + c0;
    if (prm.out_mode == Y2_OUT_BF16_PADDED) {
        if (in_range) {
            __nv_bfloat16 *o = reinterpret_cast<__nv_bfloat16 *>(prm.out) + (size_t)p * prm.out_cs + ch0;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (ch0 + q * 8 < prm.cout) {
                    uint4 w;
                    if (valid) {
                        w.x = pack_bf16x2(f[q * 8 + 0], f[q * 8 + 1]);
                        w.y = pack_bf16x2(f[q * 8 + 2], f[q * 8 + 3]);
                        w.z = pack_bf16x2(f[q * 8 + 4], f[q * 8 + 5]);
                        w.w = pack_bf16x2(f[q * 8 + 6], f[q * 8 + 7]);
                    } else {
                        w = make_uint4(0u, 0u, 0u, 0u);
                    }
                    *reinterpret_cast<uint4 *>(o + q * 8) = w;
                }
            }
        }
    } else {  // Y2_OUT_F32_FLAT: [B][h*w][out_cs]
        if (valid) {
            float *o = reinterpret_cast<float *>(prm.out) +
                       ((size_t)b * prm.h * prm.w + (size_t)y * prm.w + x) * prm.out_cs + ch0;
#pragma unroll
            for (int j = 0; j < 32; ++j)
                if (ch0 + j < prm.cout) o[j] = f[j];
        }
    }
}

// fp32 flat output [B][h*w][out_cs] of a wide head (yolo9000: 28 269 filters) through the warp's 4 KB staging tile.
// After tcgen05.ld a lane owns one output ROW, so storing from registers means 32 scalar stores per lane that touch
// 32 different lines each; staged, the warp writes 4 rows x 128 contiguous bytes per instruction (8 instructions per
// 32 x 32 chunk).  flat_row: this lane's row in the output (b*h*w + y*w + x), -1 for pad positions.  out_cs % 4 == 0.
template <int ACT>
__device__ __forceinline__ void slab_store_f32_staged(const SlabParams &prm, uint4 *stage, const uint32_t (&v)[32],
                                                      const float2 *sab, int c0, int n0, long long flat_row, int lane)
{
    const float4 *ab4 = reinterpret_cast<const float4 *>(sab + c0);
    uint32_t f[32];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const float4 q = ab4[j];  // (alpha, beta) of two filters
        float t0 = fmaf(__uint_as_float(v[2 * j]), q.x, q.y);
        float t1 = fmaf(__uint_as_float(v[2 * j + 1]), q.z, q.w);
        if (ACT == Y2_ACT_LEAKY) {
            t0 = fmaxf(t0, 0.1f * t0);
            t1 = fmaxf(t1, 0.1f * t1);
        } else if (ACT == Y2_ACT_LOGISTIC) {
            t0 = 1.f / (1.f + __expf(-t0));
            t1 = 1.f / (1.f + __expf(-t1));
        }
        f[2 * j] = __float_as_uint(t0);
        f[2 * j + 1] = __float_as_uint(t1);
    }
    __syncwarp();  // the previous chunk has been read out of the tile
#pragma unroll
    for (int c = 0; c < 8; ++c)
        stage[lane * 8 + (c ^ (lane & 7))] = make_uint4(f[4 * c], f[4 * c + 1], f[4 * c + 2], f[4 * c + 3]);
    __syncwarp();
    const int ch = n0 + c0 + (lane & 7) * 4;
    float *out = reinterpret_cast<float *>(prm.out);
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int r = it * 4 + (lane >> 3);
        const long long fr = __shfl_sync(0xffffffffu, flat_row, r);
        const uint4 q = stage[r * 8 + ((lane & 7) ^ (r & 7))];
        if (fr >= 0 && ch < prm.cout) {
            float *o = out + fr * prm.out_cs + ch;
            if (ch + 4 <= prm.cout) {
                // streaming store: 2 GB of head output per yolo9000 step must not push the 58 MB weight matrix (read
                // again for every position tile) out of the L2
                __stcs(reinterpret_cast<uint4 *>(o), q);
            } else {  // the last filters of a head whose count is not a multiple of 4
                o[0] = __uint_as_float(q.x);
                if (ch + 1 < prm.cout) o[1] = __uint_as_float(q.y);
                if (ch + 2 < prm.cout) o[2] = __uint_as_float(q.z);
            }
        }
    }
}

// affine + activation of one 32-column chunk, packed to bf16 (zeros when the row is a pad position)
template <int ACT>
__device__ __forceinline__ void slab_affine_pack(const uint32_t (&v)[32], const float2 *sab, int c0, bool valid,
                                                 uint4 *w)
{
    const float4 *ab4 = reinterpret_cast<const float4 *>(sab + c0);
    uint32_t pk[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const float4 q = ab4[j];  // (alpha, beta) of two filters
        float t0 = fmaf(__uint_as_float(v[2 * j]), q.x, q.y);
        float t1 = fmaf(__uint_as_float(v[2 * j + 1]), q.z, q.w);
        if (ACT == Y2_ACT_LEAKY) {
            t0 = fmaxf(t0, 0.1f * t0);
            t1 = fmaxf(t1, 0.1f * t1);
        } else if (ACT == Y2_ACT_LOGISTIC) {
            t0 = 1.f / (1.f + __expf(-t0));
            t1 = 1.f / (1.f + __expf(-t1));
        }
        pk[j] = valid ? pack_bf16x2(t0, t1) : 0u;
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) w[q] = make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
}

// 32 rows x 64 channels of one warp -> its 4 KB staging tile in the SWIZZLE_128B layout of the output
// tensor map (16-byte chunk c of row r at chunk c ^ (r & 7): conflict free), then ONE TMA store: the
// copy engine writes full 128-byte lines, the LSU sees 8 shared-memory stores per thread instead of 8
// global stores that touch 32 different lines each.
__device__ __forceinline__ void slab_store_tma(const void *tm_out, uint4 *stage, const uint4 (&w)[8], int lane,
                                               int p_first, int ch0)
{
    // the previous box of this warp must have been read out of the staging tile
    if (lane == 0) tma_store_wait_read();
    __syncwarp();
#pragma unroll
    for (int c = 0; c < 8; ++c) stage[lane * 8 + (c ^ (lane & 7))] = w[c];
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) {
        tma_store_2d(tm_out, stage, ch0, p_first);
        tma_store_commit();
    }
}

} // namespace y2
