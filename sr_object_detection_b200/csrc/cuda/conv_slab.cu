// Implicit-GEMM 3x3 convolution, "halo slab" variant.
//
// Replaces forward_convolutional_layer_gpu (reference convolutional_kernels.cu:77-131) for 3x3
// stride-1 'same' layers; 1x1 layers and shapes that do not fit use conv_tcgen05.cu.
//
// Why a second kernel.  In the per-tap kernel (conv_tcgen05.cu) every one of the nine taps TMA-loads
// its own shifted copy of the same activations.  Shared-memory bandwidth (TMA fill + tensor-core
// operand reads, ~128 B/clk/SM) is what bounds these layers on B200, so here
//   * the activations of a tile are loaded ONCE per channel block as a slab of consecutive flat
//     positions  [p0 - (W+1) - 1,  p0 + M + (W+1) + 1)  (padded-NHWC flat positions, see
//     yolo2_b200_kernels.h); the nine taps are nine tcgen05.mma A-descriptors whose start address
//     is shifted by  r*(W+1) + s  rows inside that slab.  The swizzle XOR is a function of the
//     absolute shared-memory address, so a row-shifted descriptor reads exactly what TMA wrote
//     (verified on B200 for SWIZZLE_128B and SWIZZLE_64B, experiments/shifted_desc_test.cu);
//   * narrow layers (<= 128 filters) use a tile of 256 positions held in TWO TMEM accumulators, so
//     every weight tile that arrives in shared memory feeds two MMAs; wide layers keep one
//     128 x 256 accumulator (the A read of an MMA is amortised over 256 filters);
//   * small weight tiles travel 3 or 9 taps per pipeline stage: the MMA-issuing thread is a single
//     latency-bound thread, one mbarrier round trip (~100 clk) per 128 tensor-pipe clocks would
//     starve the pipe;
//   * accumulators are double buffered in TMEM: the epilogue (8 warps) of tile i overlaps the MMAs
//     of tile i+1.
// The nine taps are fully unrolled and every descriptor is "base + compile-time multiple of two
// registers", so the issue loop is a few uniform-datapath adds per UTCHMMA.
//
// Warp roles (352 threads): 0 slab producer, 1 MMA issuer (+ TMEM alloc), 2 weight producer,
// 3..10 epilogue (TMEM lane quarter = warp & 3; warps 3-6 take the first half of the tile's
// accumulator columns, warps 7-10 the second half).  Producer / MMA warps run converged and
// elect one lane per issue (see elect_one_sync in y2_common.cuh).
#include "conv_epilogue.cuh"

#include <string.h>

namespace y2 {

constexpr int kSlabThreads = 352;
constexpr int kSlabEpiThreads = 256;
constexpr int kSlabMaxStagesA = 4;
constexpr int kSlabMaxStagesB = 8;

template <int BLOCK_N, int BLOCK_K, int ACCS, int TPS, int TAPS>
struct SlabCfg {
    static constexpr int kTileM = ACCS * kBlockM;
    static constexpr int kRowBytes = BLOCK_K * 2;
    static constexpr int kBBytes = BLOCK_N * BLOCK_K * 2;
    static constexpr int kBStageBytes = TPS * kBBytes;
    static constexpr int kTmemCols = (2 * ACCS * BLOCK_N <= 128) ? 128 : (2 * ACCS * BLOCK_N <= 256) ? 256 : 512;
    static_assert(2 * ACCS * BLOCK_N <= 512, "accumulators exceed TMEM");
    static_assert(TAPS == 9 || TAPS == 1, "3x3 or 1x1");
    static_assert(TAPS % TPS == 0 && (TPS == 1 || TPS == 3 || TPS == 9), "taps per stage");
    static_assert(ACCS * BLOCK_N >= 64, "each epilogue half owns whole 32-column chunks");
    static constexpr uint32_t kSBO = 8 * BLOCK_K * 2;
    static constexpr uint32_t kLayout = (BLOCK_K == 64) ? 2u : 4u;  // SWIZZLE_128B : SWIZZLE_64B
    // high word of a K-major smem descriptor: SBO>>4 at [32,46), version 1 at [46,48), swizzle [61,64)
    static constexpr uint32_t kDescHi = (kSBO >> 4) | (1u << 14) | (kLayout << 29);
    static constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) |
                                       ((uint32_t)(BLOCK_N >> 3) << 17) |
                                       ((uint32_t)(kBlockM >> 4) << 24);
};

__device__ __forceinline__ uint64_t slab_desc(uint32_t hi, uint32_t lo)
{
    return ((uint64_t)hi << 32) | (uint64_t)lo;
}

template <int BLOCK_N, int BLOCK_K, int ACCS, int TPS, int TAPS>
__global__ void __launch_bounds__(kSlabThreads, 1)
conv_slab_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                 const __grid_constant__ CUtensorMap tm_out, const __grid_constant__ SlabParams prm)
{
    using Cfg = SlabCfg<BLOCK_N, BLOCK_K, ACCS, TPS, TAPS>;
    constexpr int kTileM = Cfg::kTileM;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);

    const int stages_a = prm.stages_a, stages_b = prm.stages_b;
    uint8_t *smem_a = smem;
    uint8_t *smem_b = smem + (size_t)stages_a * prm.slab_bytes;
    uint8_t *aux = smem_b + (size_t)stages_b * Cfg::kBStageBytes;
    float2 *s_ab = reinterpret_cast<float2 *>(aux);  // [2 buf][BLOCK_N] (alpha, beta)
    uint64_t *bars = reinterpret_cast<uint64_t *>(aux + 2 * BLOCK_N * 8);
    uint64_t *a_full = bars;
    uint64_t *a_empty = bars + kSlabMaxStagesA;
    uint64_t *b_full = bars + 2 * kSlabMaxStagesA;
    uint64_t *b_empty = b_full + kSlabMaxStagesB;
    uint64_t *tfull_bar = b_empty + kSlabMaxStagesB;
    uint64_t *tempty_bar = tfull_bar + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty_bar + 2);
    // [8 epilogue warps][32 rows][128 B] staging of the TMA stores, 1024-byte aligned (swizzle atom)
    uint4 *s_stage = reinterpret_cast<uint4 *>(aux + ((2 * BLOCK_N * 8 + 512 + 1023) / 1024) * 1024);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int total_tiles = prm.tiles_m * prm.tiles_n;
    const int cblocks = prm.cblocks;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tm_a);
        tma_prefetch_desc(&tm_b);
        for (int i = 0; i < stages_a; ++i) {
            mbar_init(&a_full[i], 1);
            mbar_init(&a_empty[i], 1);
        }
        for (int i = 0; i < stages_b; ++i) {
            mbar_init(&b_full[i], 1);
            mbar_init(&b_empty[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tfull_bar[i], 1);
            mbar_init(&tempty_bar[i], kSlabEpiThreads);
        }
        fence_barrier_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                         smem_u32(tmem_slot)),
                     "r"((uint32_t)Cfg::kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    // the TMEM base is read from *tmem_slot where it is used rather than held in a register for the whole kernel:
    // the epilogue warps run at the 168-register cap

    pdl_launch_dependents();
    if (warp == 0) {
        // ===================== slab producer =====================
        pdl_wait();  // activations = the previous layer's output (weights are prefetched by warp 2 meanwhile)
        int stage = 0;
        uint32_t phase = 0;
        const uint32_t slab_tx = (uint32_t)prm.slab_loads * prm.box_rows * Cfg::kRowBytes;
        const uint32_t load_bytes = (uint32_t)prm.box_rows * Cfg::kRowBytes;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const int mq = tile / prm.tiles_n;
            const int m_tile = prm.reverse ? prm.tiles_m - 1 - mq : mq;
            const int row0 = m_tile * kTileM - prm.halo;
            for (int cb = 0; cb < cblocks; ++cb) {
                mbar_wait(&a_empty[stage], phase ^ 1, 1);
                if (elect_one_sync()) {
                    uint8_t *sa = smem_a + (size_t)stage * prm.slab_bytes;
                    mbar_expect_tx(&a_full[stage], slab_tx);
                    for (int i = 0; i < prm.slab_loads; ++i)
                        tma_load_2d(&tm_a, &a_full[stage], sa + i * load_bytes, cb * BLOCK_K,
                                    row0 + i * prm.box_rows);
                }
                __syncwarp();
                if (++stage == stages_a) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 2) {
        // ===================== weight producer =====================
        int stage = 0;
        uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const int mq = tile / prm.tiles_n;
            const int m_tile = prm.reverse ? prm.tiles_m - 1 - mq : mq;
            const int n0 = (tile - mq * prm.tiles_n) * BLOCK_N;
            for (int cb = 0; cb < cblocks; ++cb) {
#pragma unroll 1
                for (int g = 0; g < TAPS / TPS; ++g) {
                    mbar_wait(&b_empty[stage], phase ^ 1, 2);
                    if (elect_one_sync()) {
                        uint8_t *sb = smem_b + (size_t)stage * Cfg::kBStageBytes;
                        mbar_expect_tx(&b_full[stage], (uint32_t)Cfg::kBStageBytes);
#pragma unroll
                        for (int t = 0; t < TPS; ++t)
                            tma_load_2d(&tm_b, &b_full[stage], sb + t * Cfg::kBBytes,
                                        ((g * TPS + t) * cblocks + cb) * BLOCK_K, n0);
                    }
                    __syncwarp();
                    if (++stage == stages_b) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        int sa_i = 0, sb_i = 0;
        uint32_t pa = 0, pb = 0;
        int it = 0;
        // descriptor low words (address >> 4, LBO field = 1) and their strides, all in 16-byte units
        const uint32_t a_lo0 = ((smem_u32(smem_a) & 0x3FFFFu) >> 4) | (1u << 16);
        const uint32_t b_lo0 = ((smem_u32(smem_b) & 0x3FFFFu) >> 4) | (1u << 16);
        const uint32_t slab16 = (uint32_t)prm.slab_bytes >> 4;
        constexpr uint32_t kRow16 = Cfg::kRowBytes >> 4;        // one position (row) of the slab
        const uint32_t wp16 = (uint32_t)prm.wp * kRow16;        // one image row of the slab
        constexpr uint32_t kAcc16 = kBlockM * kRow16;           // second accumulator: +128 positions
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
            const int buf = it & 1;
            const uint32_t buf_phase = (it >> 1) & 1;
            mbar_wait(&tempty_bar[buf], buf_phase ^ 1, 3);
            tc_fence_after();
            const uint32_t d0 = *tmem_slot + (uint32_t)(buf * ACCS * BLOCK_N);
            for (int cb = 0; cb < cblocks; ++cb) {
                mbar_wait(&a_full[sa_i], pa, 4);
                const uint32_t a_lo = a_lo0 + (uint32_t)sa_i * slab16;
                const uint32_t acc_first = cb != 0;  // tap 0, k 0 of block 0 overwrites the accumulator
#pragma unroll
                for (int tap = 0; tap < TAPS; ++tap) {
                    if (tap % TPS == 0) {
                        mbar_wait(&b_full[sb_i], pb, 5);
                        tc_fence_after();
                    }
                    if (elect_one_sync()) {
                        const uint32_t b_lo = b_lo0 + (uint32_t)sb_i * (Cfg::kBStageBytes >> 4) +
                                              (uint32_t)(tap % TPS) * (Cfg::kBBytes >> 4);
                        const uint32_t a_tap = a_lo + (uint32_t)(tap / 3) * wp16 + (uint32_t)(tap % 3) * kRow16;
#pragma unroll
                        for (int a = 0; a < ACCS; ++a) {
#pragma unroll
                            for (int k = 0; k < BLOCK_K / 16; ++k)
                                umma_bf16(d0 + (uint32_t)(a * BLOCK_N),
                                          slab_desc(Cfg::kDescHi, a_tap + (uint32_t)a * kAcc16 + (uint32_t)(k * 2)),
                                          slab_desc(Cfg::kDescHi, b_lo + (uint32_t)(k * 2)), Cfg::kIdesc,
                                          (tap == 0 && k == 0) ? acc_first : 1u);
                        }
                        if (tap % TPS == TPS - 1) umma_commit(&b_empty[sb_i]);
                        if (tap == TAPS - 1) {
                            umma_commit(&a_empty[sa_i]);
                            if (cb == cblocks - 1) umma_commit(&tfull_bar[buf]);
                        }
                    }
                    __syncwarp();
                    if (tap % TPS == TPS - 1) {
                        if (++sb_i == stages_b) { sb_i = 0; pb ^= 1; }
                    }
                }
                if (++sa_i == stages_a) { sa_i = 0; pa ^= 1; }
            }
        }
    } else {
        // ===================== epilogue (warps 3..10) =====================
        const int quarter = warp & 3;
        const int half = (warp - 3) >> 2;
        const int et = threadIdx.x - 96;  // 0..255
        // this warp's share of the tile: with two accumulators, warps 3-6 drain the first and warps
        // 7-10 the second; with one, each group drains half of its columns
        constexpr int kSpan = ACCS * BLOCK_N / 2;
        const int acc = (ACCS == 2) ? half : 0;
        const int col0 = (ACCS == 2) ? 0 : half * kSpan;
        const int img_pos = prm.hp * prm.wp;
        const bool ab_lane = et < BLOCK_N;
        int it = 0;
        // (alpha, beta) of the first tile; later tiles are prefetched one tile ahead
        if ((int)blockIdx.x < total_tiles && ab_lane) {
            const int n0 = ((int)blockIdx.x % prm.tiles_n) * BLOCK_N;
            s_ab[et] = make_float2(__ldg(prm.alpha + n0 + et), __ldg(prm.beta + n0 + et));
        }
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
            const int buf = it & 1;
            const uint32_t buf_phase = (it >> 1) & 1;
            const int mq = tile / prm.tiles_n;
            const int m_tile = prm.reverse ? prm.tiles_m - 1 - mq : mq;
            const int n0 = (tile - mq * prm.tiles_n) * BLOCK_N;
            const float2 *sab = s_ab + (prm.tiles_n > 1 ? buf * BLOCK_N : 0);
            // one filter block per layer: (alpha, beta) never change and the epilogue warps stay decoupled
            const bool reload = prm.tiles_n > 1 || it == 0 || prm.couple;
            if (reload) asm volatile("bar.sync 1, 256;" ::: "memory");  // sab[buf] written, sab[buf^1] free
            const int next = tile + (int)gridDim.x;
            float2 ab_next = make_float2(1.f, 0.f);
            if (prm.tiles_n > 1 && next < total_tiles && ab_lane) {
                const int nn = (next % prm.tiles_n) * BLOCK_N;
                ab_next = make_float2(__ldg(prm.alpha + nn + et), __ldg(prm.beta + nn + et));
            }
            const int p = m_tile * kTileM + acc * kBlockM + quarter * 32 + lane;
            const bool in_range = p < prm.total_pos;
            const int b = p / img_pos;
            const int rem = p - b * img_pos;
            const int y = rem / prm.wp;
            const int x = rem - y * prm.wp;
            const bool valid = in_range && (y < prm.h) && (x < prm.w);
            const uint32_t taddr = *tmem_slot + ((uint32_t)(quarter * 32) << 16) +
                                   (uint32_t)((buf * ACCS + acc) * BLOCK_N + col0);

            mbar_wait(&tfull_bar[buf], buf_phase, 6);
            tc_fence_after();
            if constexpr (kSpan >= 64) {
#pragma unroll 1
                for (int c = 0; c < kSpan; c += 64) {
                    uint32_t v0[32], v1[32];
                    tmem_ld32(taddr + (uint32_t)c, v0);
                    tmem_ld32(taddr + (uint32_t)(c + 32), v1);
                    tmem_ld_wait();
                    if (c + 64 >= kSpan) {  // accumulator drained into registers: hand it back to the MMA warp
                        tc_fence_before();
                        mbar_arrive(&tempty_bar[buf]);
                    }
                    if (prm.tma_store == 2) {  // fp32 flat head: staged, row-contiguous 16-byte stores
                        const long long fr = valid ? ((long long)b * prm.h + y) * prm.w + x : -1ll;
                        uint4 *st = s_stage + (warp - 3) * 256;
                        if (prm.act == Y2_ACT_LINEAR) {
                            slab_store_f32_staged<Y2_ACT_LINEAR>(prm, st, v0, sab, col0 + c, n0, fr, lane);
                            slab_store_f32_staged<Y2_ACT_LINEAR>(prm, st, v1, sab, col0 + c + 32, n0, fr, lane);
                        } else if (prm.act == Y2_ACT_LEAKY) {
                            slab_store_f32_staged<Y2_ACT_LEAKY>(prm, st, v0, sab, col0 + c, n0, fr, lane);
                            slab_store_f32_staged<Y2_ACT_LEAKY>(prm, st, v1, sab, col0 + c + 32, n0, fr, lane);
                        } else {
                            slab_store_f32_staged<Y2_ACT_LOGISTIC>(prm, st, v0, sab, col0 + c, n0, fr, lane);
                            slab_store_f32_staged<Y2_ACT_LOGISTIC>(prm, st, v1, sab, col0 + c + 32, n0, fr, lane);
                        }
                    } else if (prm.tma_store) {  // bf16 tensor, 64-channel aligned: staged, one TMA store per warp
                        uint4 w[8];
                        if (prm.act == Y2_ACT_LEAKY) {
                            slab_affine_pack<Y2_ACT_LEAKY>(v0, sab, col0 + c, valid, w);
                            slab_affine_pack<Y2_ACT_LEAKY>(v1, sab, col0 + c + 32, valid, w + 4);
                        } else if (prm.act == Y2_ACT_LINEAR) {
                            slab_affine_pack<Y2_ACT_LINEAR>(v0, sab, col0 + c, valid, w);
                            slab_affine_pack<Y2_ACT_LINEAR>(v1, sab, col0 + c + 32, valid, w + 4);
                        } else {
                            slab_affine_pack<Y2_ACT_LOGISTIC>(v0, sab, col0 + c, valid, w);
                            slab_affine_pack<Y2_ACT_LOGISTIC>(v1, sab, col0 + c + 32, valid, w + 4);
                        }
                        slab_store_tma(&tm_out, s_stage + (warp - 3) * 256, w, lane, p - lane, n0 + col0 + c);
                    } else if (prm.act == Y2_ACT_LEAKY) {
                        slab_epilogue_chunk<Y2_ACT_LEAKY>(prm, v0, sab, col0 + c, n0, p, b, y, x, in_range, valid);
                        slab_epilogue_chunk<Y2_ACT_LEAKY>(prm, v1, sab, col0 + c + 32, n0, p, b, y, x, in_range, valid);
                    } else if (prm.act == Y2_ACT_LINEAR) {
                        slab_epilogue_chunk<Y2_ACT_LINEAR>(prm, v0, sab, col0 + c, n0, p, b, y, x, in_range, valid);
                        slab_epilogue_chunk<Y2_ACT_LINEAR>(prm, v1, sab, col0 + c + 32, n0, p, b, y, x, in_range, valid);
                    } else {
                        slab_epilogue_chunk<Y2_ACT_LOGISTIC>(prm, v0, sab, col0 + c, n0, p, b, y, x, in_range, valid);
                        slab_epilogue_chunk<Y2_ACT_LOGISTIC>(prm, v1, sab, col0 + c + 32, n0, p, b, y, x, in_range, valid);
                    }
                }
            } else {  // BLOCK_N == 32, two accumulators: one 32-column chunk per warp
                uint32_t v0[32];
                tmem_ld32(taddr, v0);
                tmem_ld_wait();
                tc_fence_before();
                mbar_arrive(&tempty_bar[buf]);
                if (prm.act == Y2_ACT_LEAKY)
                    slab_epilogue_chunk<Y2_ACT_LEAKY>(prm, v0, sab, col0, n0, p, b, y, x, in_range, valid);
                else if (prm.act == Y2_ACT_LINEAR)
                    slab_epilogue_chunk<Y2_ACT_LINEAR>(prm, v0, sab, col0, n0, p, b, y, x, in_range, valid);
                else
                    slab_epilogue_chunk<Y2_ACT_LOGISTIC>(prm, v0, sab, col0, n0, p, b, y, x, in_range, valid);
            }
            if (prm.tiles_n > 1 && next < total_tiles && ab_lane) s_ab[(buf ^ 1) * BLOCK_N + et] = ab_next;
        }
        if (prm.tma_store == 1 && lane == 0) tma_store_wait_all();  // the copies read this CTA's shared memory
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(*tmem_slot),
                     "r"((uint32_t)Cfg::kTmemCols)
                     : "memory");
    }
}

// -------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------
// (BLOCK_N, BLOCK_K, ACCS, TPS, TAPS): 3x3 layers with weight stages of 16-36 KB, then the 1x1 layers
#define Y2_FOR_EACH_SLAB_CFG(X)                                                                          \
    X(256, 64, 1, 1, 9) X(128, 64, 2, 1, 9) X(64, 64, 2, 3, 9) X(32, 64, 2, 9, 9) X(256, 32, 1, 1, 9)      \
    X(128, 32, 2, 3, 9) X(64, 32, 2, 9, 9) X(32, 32, 2, 9, 9) X(256, 64, 1, 1, 1) X(128, 64, 2, 1, 1)    \
    X(64, 64, 2, 1, 1) X(32, 64, 2, 1, 1) X(128, 32, 2, 1, 1) X(64, 32, 2, 1, 1) X(32, 32, 2, 1, 1)

static int slab_tps(int bn, int bk, int taps)
{
#define Y2_CASE(BN, BK, ACCS, TPS, TAPS) \
    if (bn == BN && bk == BK && taps == TAPS) return TPS;
    Y2_FOR_EACH_SLAB_CFG(Y2_CASE)
#undef Y2_CASE
    return 0;
}

template <int BN, int BK, int ACCS, int TPS, int TAPS>
static int slab_prepare_cfg()
{
    static bool attr_done[64] = {false};
    int dev = 0;
    Y2_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && !attr_done[dev]) {
        Y2_CUDA_CHECK(cudaFuncSetAttribute(conv_slab_kernel<BN, BK, ACCS, TPS, TAPS>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        attr_done[dev] = true;
    }
    return Y2_OK;
}

int slab_plan_init(y2_conv_plan *pl, const y2_conv_desc *d, ConvChoice choice)
{
    const int taps = d->ksize * d->ksize;
    const int bn = d->block_n;
    const int accs = bn == 256 ? 1 : 2;
    const int tile_m = accs * kBlockM;
    const int bk = d->block_k;
    const int tps = slab_tps(bn, bk, taps);
    if (!tps || d->npad % bn) return Y2_EINVAL;
    const int hp = d->h + 1, wp = d->w + 1;
    const long long total = (long long)d->batch * hp * wp;
    const int row_bytes = bk * 2;
    const int halo = taps == 9 ? wp + 1 : 0;
    const int slab_rows = tile_m + 2 * halo;
    const int loads = (slab_rows + 255) / 256;
    int box_rows = (slab_rows + loads - 1) / loads;
    // a load must cover whole swizzle atoms (1024 bytes: 8 rows of 128 bytes, 16 rows of 64 bytes)
    const int gran = 1024 / row_bytes;
    box_rows = (box_rows + gran - 1) / gran * gran;
    if (box_rows > 256) return Y2_EINVAL;
    const int slab_bytes = loads * box_rows * row_bytes;  // multiple of 1024
    const int b_stage = tps * bn * bk * 2;
    const int aux = ((2 * bn * 8 + 512 + 1023) / 1024) * 1024 + 8 * 4096;  // alpha/beta, barriers | store staging
    const int budget = 227 * 1024 - 1024 - aux;
    // 1x1: every channel block needs a fresh slab, keep as many slabs as weight tiles in flight
    int stages_a = 2;
    if (taps == 1) {
        stages_a = budget / (slab_bytes + b_stage);
        if (stages_a > kSlabMaxStagesA) stages_a = kSlabMaxStagesA;
        if (stages_a < 2) return Y2_EINVAL;
    }
    int stages_b = (budget - stages_a * slab_bytes) / b_stage;
    if (stages_b > kSlabMaxStagesB) stages_b = kSlabMaxStagesB;
    // wide images (yolo.cfg at 608: 152-position rows) leave room for two weight stages only: still well ahead
    // of the per-tap kernel, which reloads the activations for every tap
    if (stages_b < 2 || (tps == 1 && stages_b < 3 && wp <= 128)) return Y2_EINVAL;
    const int ktot = taps * d->cin;
    int rc = encode_2d_bf16(&pl->tm_a, d->in, (uint64_t)d->cin, (uint64_t)total, (uint64_t)d->in_cs * 2,
                            (uint32_t)bk, (uint32_t)box_rows, bk);
    if (rc == Y2_OK)
        rc = encode_2d_bf16(&pl->tm_b, d->wt, (uint64_t)ktot, (uint64_t)d->npad, (uint64_t)ktot * 2, (uint32_t)bk,
                            (uint32_t)bn, bk);
    if (rc != Y2_OK) return rc;
    SlabParams &p = pl->slab;
    // output through TMA stores when it is the bf16 tensor in whole 64-channel groups (box = 64 channels x 32
    // positions, SWIZZLE_128B): pad positions are stored as zeros like before, rows past the tensor are clipped
    p.tma_store = 0;
    memset(&pl->tm_out, 0, sizeof(pl->tm_out));
    if (d->out_mode == Y2_OUT_BF16_PADDED && bn >= 64 && d->cout % 64 == 0) {
        rc = encode_2d_bf16(&pl->tm_out, d->out, (uint64_t)d->cout, (uint64_t)total, (uint64_t)d->out_cs * 2, 64u, 32u, 64);
        if (rc != Y2_OK) return rc;
        p.tma_store = 1;
    }
    // fp32 heads with 16-byte aligned rows: staged row-contiguous stores (conv_epilogue.cuh) instead of 32 scalar
    // stores per lane and chunk
    const bool f32_staged = d->out_mode == Y2_OUT_F32_FLAT && bn >= 128 && d->out_cs % 4 == 0 &&
                            ((uintptr_t)d->out & 15) == 0;
    if (f32_staged) p.tma_store = 2;
    p.cblocks = d->cin / bk;
    p.wp = wp;
    p.hp = hp;
    p.h = d->h;
    p.w = d->w;
    p.total_pos = (int)total;
    p.tiles_m = (int)((total + tile_m - 1) / tile_m);
    p.tiles_n = d->npad / bn;
    p.halo = halo;
    p.slab_loads = loads;
    p.box_rows = box_rows;
    p.slab_bytes = slab_bytes;
    p.stages_a = stages_a;
    p.stages_b = stages_b;
    p.cout = d->cout;
    p.act = d->act;
    p.out_mode = d->out_mode;
    p.out_cs = d->out_cs;
    p.alpha = d->alpha;
    p.beta = d->beta;
    p.out = d->out;
    // measured on B200: lock-stepped epilogue warps write 128-byte rows (<= 64 filters) 10% faster, wider
    // rows prefer free-running warps
    p.couple = bn <= 64;
    // A layer reads what the layer before it has just written, first position first.  When that tensor is
    // about as large as the 126 MB L2 (or larger: yolo-voc L5 at batch 64 reads 180 MB), only its most
    // recently written end is still resident - so walk the position tiles last-to-first and take that part
    // from the L2.  Measured at batch 64 (A/B of the whole step, same box): L9 (92 MB in) 34 -> 31 us, the
    // step -1.0 %; layers with <= 48 MB inputs are all-L2 either way (L13: 25 -> 27 us reversed), hence the
    // threshold.
    // The producer may itself have walked last-to-first (in_order 1): then the resident end is the front.
    p.reverse = (double)d->batch * hp * wp * d->in_cs * 2.0 > 64e6 && !d->in_order;
    pl->variant = kVariantSlab;
    pl->block_n = bn;
    pl->block_k = bk;
    pl->smem_bytes = (size_t)stages_a * slab_bytes + (size_t)stages_b * b_stage + aux + 1024;
    const int tiles = p.tiles_m * p.tiles_n;
    const int sms = sm_count();
    // 1x1 layers: the 256-position tiles pay off only while every SM still gets two or more of them and
    // the output is the bf16 tensor (measured on B200: L5/L9/L13 +5..15%, the 13x13 layers and the fp32
    // head are faster on the per-tap kernel's 128-position tiles)
    if (taps == 1 && !f32_staged && (tiles < 2 * sms || d->out_mode != Y2_OUT_BF16_PADDED) && choice == kChooseAuto)
        return Y2_EINVAL;
    pl->grid = tiles < sms ? tiles : sms;
    pl->taps = taps;
#define Y2_CASE(BN, BK, ACCS, TPS, TAPS) \
    if (bn == BN && bk == BK && taps == TAPS) return slab_prepare_cfg<BN, BK, ACCS, TPS, TAPS>();
    Y2_FOR_EACH_SLAB_CFG(Y2_CASE)
#undef Y2_CASE
    return Y2_EINVAL;
}

int slab_plan_launch(const y2_conv_plan *pl, cudaStream_t st)
{
#define Y2_CASE(BN, BK, ACCS, TPS, TAPS)                                                                       \
    if (pl->block_n == BN && pl->block_k == BK && pl->taps == TAPS) {                                            \
        Y2_CUDA_CHECK(launch_pdl(conv_slab_kernel<BN, BK, ACCS, TPS, TAPS>, dim3(pl->grid), dim3(kSlabThreads),         \
                                 pl->smem_bytes, st, pl->tm_a, pl->tm_b, pl->tm_out, pl->slab));                         \
        Y2_LAUNCH_CHECK();                                                                                       \
        return Y2_OK;                                                                                            \
    }
    Y2_FOR_EACH_SLAB_CFG(Y2_CASE)
#undef Y2_CASE
    set_error("slab_plan_launch: no kernel for block_n=%d block_k=%d", pl->block_n, pl->block_k);
    return Y2_EINVAL;
}

} // namespace y2
