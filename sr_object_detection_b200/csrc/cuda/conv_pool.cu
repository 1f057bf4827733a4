// 3x3 convolution + batchnorm + leaky-ReLU fused with the 2x2/2 maxpool that follows it.
//
// Replaces forward_convolutional_layer_gpu (reference convolutional_kernels.cu:77-131) AND the
// forward_maxpool_layer_gpu behind it (maxpool_layer_kernels.cu:10-48, 87-97) for the early layers
// of every north-star cfg (yolo-voc L2+L3: 32 -> 64 @208, L6+L7: 64 -> 128 @104): the
// full-resolution activation - the largest tensor of the network, 354 MB at batch 64 - is never
// written or re-read; only the pooled tensor leaves the SM.
//
// Geometry.  A patch of (R+2) input rows x P positions (P = tile width + 2) of one image is loaded
// by ONE 3-D TMA box from the padded-NHWC tensor (out-of-image rows / columns arrive as zeros or as
// the stored zero pads) and sits densely in shared memory, flat row = r*P + q.  Image row i of the
// patch is the MMA operand of 128 consecutive flat rows starting at (i + dr)*P + ds for tap (dr, ds)
// - the same row-shifted-descriptor trick as conv_slab.cu, here on a 2-D patch, so that the two
// accumulators of a slot hold image rows y and y+1 in the SAME TMEM lanes (lanes >= tile width are
// junk and discarded).  The 2x2 pool is then a vertical max inside a thread and one shuffle with the
// neighbouring lane; each lane of a pair finishes half of the channels (affine, leaky, bf16, store).
// max before the affine map is exact: the host makes every alpha_f >= 0 (see stem_tcgen05.cu).
//
// Restricted to one channel block (C_in <= 64) and 64 / 128 filters; weights are streamed per row
// pair exactly like conv_slab.cu streams them per tile.
//
// Warp roles (608 threads): 0 patch producer, 1 MMA issuer (+ TMEM alloc), 2 weight producer,
// 3..18 epilogue: four groups of four warps = (row-pair parity) x (half of every 32-channel chunk);
// the epilogue is a long dependent chain per thread, so it is spread over many warps.
#include "conv_plan.cuh"

namespace y2 {

constexpr int kPoolThreads = 608;  // 3 producer / MMA warps + 16 epilogue warps
constexpr int kPoolMaxStagesB = 8;
constexpr int kPoolStagesA = 2;

template <int BLOCK_N, int BLOCK_K, int TPS>
struct PoolCfg {
    static constexpr int kRowBytes = BLOCK_K * 2;
    static constexpr int kBBytes = BLOCK_N * BLOCK_K * 2;
    static constexpr int kBStageBytes = TPS * kBBytes;
    static constexpr int kSlotCols = 2 * BLOCK_N;              // two accumulators: image rows y, y+1
    static constexpr int kSlots = 512 / kSlotCols;             // 4 (N = 64) or 2 (N = 128)
    static_assert(BLOCK_N == 64 || BLOCK_N == 128, "filters per tile");
    static_assert(9 % TPS == 0, "taps per stage");
    static constexpr uint32_t kSBO = 8 * BLOCK_K * 2;
    static constexpr uint32_t kLayout = (BLOCK_K == 64) ? 2u : 4u;  // SWIZZLE_128B : SWIZZLE_64B
    static constexpr uint32_t kDescHi = (kSBO >> 4) | (1u << 14) | (kLayout << 29);
    static constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BLOCK_N >> 3) << 17) |
                                       ((uint32_t)(kBlockM >> 4) << 24);
};

__device__ __forceinline__ void tma_load_3d_bf16(const void *desc, uint64_t *bar, void *smem_dst, int c0, int c1, int c2)
{
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(smem_dst)),
        "l"(desc), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

template <int BLOCK_N, int BLOCK_K, int TPS>
__global__ void __launch_bounds__(kPoolThreads, 1)
conv_pool_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                 const PoolParams prm)
{
    using Cfg = PoolCfg<BLOCK_N, BLOCK_K, TPS>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);

    const int stages_b = prm.stages_b;
    uint8_t *smem_a = smem;
    uint8_t *smem_b = smem + (size_t)kPoolStagesA * prm.patch_bytes;  // also the landing zone of junk-lane reads
    uint8_t *aux = smem_b + (size_t)stages_b * Cfg::kBStageBytes;
    float2 *s_ab = reinterpret_cast<float2 *>(aux);  // [BLOCK_N] (alpha, beta)
    uint64_t *bars = reinterpret_cast<uint64_t *>(aux + BLOCK_N * 8);
    uint64_t *a_full = bars;
    uint64_t *a_empty = bars + kPoolStagesA;
    uint64_t *b_full = bars + 2 * kPoolStagesA;
    uint64_t *b_empty = b_full + kPoolMaxStagesB;
    uint64_t *tfull_bar = b_empty + kPoolMaxStagesB;
    uint64_t *tempty_bar = tfull_bar + Cfg::kSlots;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty_bar + Cfg::kSlots);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int P = prm.wt + 2;
    const int pairs = prm.rows / 2;  // row pairs per patch
    const int per_img = prm.tiles_x * prm.tiles_y;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tm_a);
        tma_prefetch_desc(&tm_b);
        for (int i = 0; i < kPoolStagesA; ++i) {
            mbar_init(&a_full[i], 1);
            mbar_init(&a_empty[i], 1);
        }
        for (int i = 0; i < stages_b; ++i) {
            mbar_init(&b_full[i], 1);
            mbar_init(&b_empty[i], 1);
        }
        for (int i = 0; i < Cfg::kSlots; ++i) {
            mbar_init(&tfull_bar[i], 1);
            mbar_init(&tempty_bar[i], 256);  // both channel-half groups
        }
        fence_barrier_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (threadIdx.x >= 96 && threadIdx.x - 96 < BLOCK_N) {
        const int f = threadIdx.x - 96;
        s_ab[f] = make_float2(__ldg(prm.alpha + f), __ldg(prm.beta + f));
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    pdl_launch_dependents();
    if (warp == 0) {
        // ===================== patch producer: one 3-D TMA box per tile =====================
        pdl_wait();  // activations = the previous layer's output (weights are prefetched by warp 2 meanwhile)
        int it = 0;
        for (int tile = blockIdx.x; tile < prm.total_tiles; tile += gridDim.x, ++it) {
            const int s = it & 1;
            const uint32_t ph = (uint32_t)(it >> 1) & 1u;
            const int vt = prm.reverse ? prm.total_tiles - 1 - tile : tile;
            const int b = vt / per_img;
            const int t = vt - b * per_img;
            const int ty = t / prm.tiles_x, tx = t - ty * prm.tiles_x;
            mbar_wait(&a_empty[s], ph ^ 1, 1);
            if (elect_one_sync()) {
                mbar_expect_tx(&a_full[s], (uint32_t)((prm.rows + 2) * P * Cfg::kRowBytes));
                tma_load_3d_bf16(&tm_a, &a_full[s], smem_a + (size_t)s * prm.patch_bytes, 0, tx * prm.wt - 1,
                                 b * (prm.h + 1) + ty * prm.rows - 1);
            }
            __syncwarp();
        }
    } else if (warp == 2) {
        // ===================== weight producer: all nine taps for every row pair =====================
        int stage = 0;
        uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < prm.total_tiles; tile += gridDim.x) {
            for (int j = 0; j < pairs; ++j) {
#pragma unroll 1
                for (int g = 0; g < 9 / TPS; ++g) {
                    mbar_wait(&b_empty[stage], phase ^ 1, 2);
                    if (elect_one_sync()) {
                        uint8_t *sb = smem_b + (size_t)stage * Cfg::kBStageBytes;
                        mbar_expect_tx(&b_full[stage], (uint32_t)Cfg::kBStageBytes);
#pragma unroll
                        for (int t = 0; t < TPS; ++t)
                            tma_load_2d(&tm_b, &b_full[stage], sb + t * Cfg::kBBytes, (g * TPS + t) * BLOCK_K, 0);
                    }
                    __syncwarp();
                    if (++stage == stages_b) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        int sb_i = 0;
        uint32_t pb = 0;
        int it = 0, slot_it = 0;
        const uint32_t a_lo0 = ((smem_u32(smem_a) & 0x3FFFFu) >> 4) | (1u << 16);
        const uint32_t b_lo0 = ((smem_u32(smem_b) & 0x3FFFFu) >> 4) | (1u << 16);
        const uint32_t patch16 = (uint32_t)prm.patch_bytes >> 4;
        constexpr uint32_t kRow16 = Cfg::kRowBytes >> 4;
        const uint32_t p16 = (uint32_t)P * kRow16;  // one patch row
        for (int tile = blockIdx.x; tile < prm.total_tiles; tile += gridDim.x, ++it) {
            const int s = it & 1;
            mbar_wait(&a_full[s], (uint32_t)(it >> 1) & 1u, 4);
            const uint32_t a_lo = a_lo0 + (uint32_t)s * patch16;
            for (int j = 0; j < pairs; ++j, ++slot_it) {
                const int slot = slot_it % Cfg::kSlots;
                mbar_wait(&tempty_bar[slot], ((uint32_t)(slot_it / Cfg::kSlots) & 1u) ^ 1u, 3);
                tc_fence_after();
                const uint32_t d0 = tmem_base + (uint32_t)(slot * Cfg::kSlotCols);
                const uint32_t a_row = a_lo + (uint32_t)(2 * j) * p16;  // image row 2j of the patch, tap row 0
#pragma unroll
                for (int tap = 0; tap < 9; ++tap) {
                    if (tap % TPS == 0) {
                        mbar_wait(&b_full[sb_i], pb, 5);
                        tc_fence_after();
                    }
                    if (elect_one_sync()) {
                        const uint32_t b_lo = b_lo0 + (uint32_t)sb_i * (Cfg::kBStageBytes >> 4) +
                                              (uint32_t)(tap % TPS) * (Cfg::kBBytes >> 4);
                        const uint32_t a_tap = a_row + (uint32_t)(tap / 3) * p16 + (uint32_t)(tap % 3) * kRow16;
#pragma unroll
                        for (int a = 0; a < 2; ++a) {  // accumulator a = image row 2j + a: one patch row further
#pragma unroll
                            for (int k = 0; k < BLOCK_K / 16; ++k)
                                umma_bf16(d0 + (uint32_t)(a * BLOCK_N),
                                          ((uint64_t)Cfg::kDescHi << 32) | (uint64_t)(a_tap + (uint32_t)a * p16 + (uint32_t)(k * 2)),
                                          ((uint64_t)Cfg::kDescHi << 32) | (uint64_t)(b_lo + (uint32_t)(k * 2)), Cfg::kIdesc,
                                          (tap == 0 && k == 0) ? 0u : 1u);
                        }
                        if (tap % TPS == TPS - 1) umma_commit(&b_empty[sb_i]);
                        if (tap == 8) {
                            umma_commit(&tfull_bar[slot]);
                            if (j == pairs - 1) umma_commit(&a_empty[s]);
                        }
                    }
                    __syncwarp();
                    if (tap % TPS == TPS - 1) {
                        if (++sb_i == stages_b) { sb_i = 0; pb ^= 1; }
                    }
                }
            }
        }
    } else {
        // ===================== epilogue: 2x2 max, affine, leaky, store =====================
        const int ew = warp - 3;             // 0..15
        const int pgroup = ew >> 3;          // row pairs alternate between the two pair groups
        const int chalf = (ew >> 2) & 1;     // columns [16 chalf, 16 chalf + 16) of every 32-column chunk
        const int quarter = warp & 3;
        const int m = quarter * 32 + lane;   // TMEM lane == position inside the tile row
        const int hsel = lane & 1;           // even lane finishes 8 of those channels, odd lane the other 8
        const int cbase = chalf * 16 + hsel * 8;
        // 64-filter layers: this thread's 16 (alpha, beta) pairs live in registers, so the epilogue leaves
        // the shared-memory pipe to the tensor core's operand reads (ncu on L2: LSU 12 % + tensor 70 % of it)
        constexpr bool kAbRegs = BLOCK_N == 64;
        float4 abr[kAbRegs ? 8 : 1];
        if (kAbRegs) {
#pragma unroll
            for (int q = 0; q < 8; ++q)
                abr[q] = reinterpret_cast<const float4 *>(s_ab + (q >> 2) * 32 + cbase)[q & 3];
        }
        int it = 0;
        // (image, tile row, tile column) advance by a constant stride: carry-propagate instead of dividing
        const int vt0 = prm.reverse ? prm.total_tiles - 1 - (int)blockIdx.x : (int)blockIdx.x;
        int b = vt0 / per_img;
        int ty = (vt0 - b * per_img) / prm.tiles_x;
        int tx = vt0 - b * per_img - ty * prm.tiles_x;
        const int db = (int)gridDim.x / per_img;
        const int dty = ((int)gridDim.x - db * per_img) / prm.tiles_x;
        const int dtx = (int)gridDim.x - db * per_img - dty * prm.tiles_x;
        for (int tile = blockIdx.x; tile < prm.total_tiles; tile += gridDim.x, ++it) {
            if (it && !prm.reverse) {
                tx += dtx;
                if (tx >= prm.tiles_x) { tx -= prm.tiles_x; ++ty; }
                ty += dty;
                if (ty >= prm.tiles_y) { ty -= prm.tiles_y; ++b; }
                b += db;
            } else if (it) {
                tx -= dtx;
                if (tx < 0) { tx += prm.tiles_x; --ty; }
                ty -= dty;
                if (ty < 0) { ty += prm.tiles_y; --b; }
                b -= db;
            }
            // A pair group owns the TMEM slots of its parity for the whole kernel (kSlots is even, so the slot
            // parity is the parity of the running row-pair count): every phase of a slot's barriers is seen
            // by the same 256 threads.  Splitting by j instead lets a group return to a slot whose previous
            // phase - drained by the other group - it never waited for, and a parity wait then passes one
            // phase early (row-pair counts per patch that are odd; hung tiny-yolo-voc at batch 64).
            for (int j = (it * pairs + pgroup) & 1; j < pairs; j += 2) {
                const int slot_it = it * pairs + j;
                const int slot = slot_it % Cfg::kSlots;
                mbar_wait_relaxed(&tfull_bar[slot], (uint32_t)(slot_it / Cfg::kSlots) & 1u, 6);
                tc_fence_after();
                const int oy = (ty * prm.rows >> 1) + j;
                const int ox = (tx * prm.wt + m) >> 1;
                const bool ok = m < prm.wt && oy < prm.oh && ox < prm.ow;
                __nv_bfloat16 *o = prm.out + (((size_t)b * (prm.oh + 1) + oy) * (prm.ow + 1) + ox) * prm.out_cs + cbase;
                const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) +
                                       (uint32_t)(slot * Cfg::kSlotCols + chalf * 16);
#pragma unroll(kAbRegs ? 2 : 1)
                for (int c0 = 0; c0 < BLOCK_N; c0 += 32) {
                    uint32_t v[16], u[16];
                    tmem_ld16(taddr + (uint32_t)c0, v);
                    tmem_ld16(taddr + (uint32_t)(BLOCK_N + c0), u);
                    tmem_ld_wait();
                    if (c0 + 32 >= BLOCK_N) {  // this thread's share of the slot is in registers
                        tc_fence_before();
                        mbar_arrive(&tempty_bar[slot]);
                    }
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
                    if (ok) {
                        const float4 *ab4 = reinterpret_cast<const float4 *>(s_ab + c0 + cbase);
                        uint32_t pk[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const float4 ab = kAbRegs ? abr[(c0 >> 5) * 4 + q] : ab4[q];  // (alpha, beta) of two filters
                            float y0 = fmaf(mx[2 * q], ab.x, ab.y);
                            float y1 = fmaf(mx[2 * q + 1], ab.z, ab.w);
                            if (prm.act == Y2_ACT_LEAKY) {
                                y0 = fmaxf(y0, 0.1f * y0);
                                y1 = fmaxf(y1, 0.1f * y1);
                            }
                            pk[q] = pack_bf16x2(y0, y1);
                        }
                        *reinterpret_cast<uint4 *>(o + c0) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                    }
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// -------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------
// (BLOCK_N, BLOCK_K, TPS)
#define Y2_FOR_EACH_POOL_CFG(X) X(64, 32, 9) X(64, 64, 3) X(128, 32, 3) X(128, 64, 1)

static int pool_tps(int bn, int bk)
{
#define Y2_CASE(BN, BK, TPS) \
    if (bn == BN && bk == BK) return TPS;
    Y2_FOR_EACH_POOL_CFG(Y2_CASE)
#undef Y2_CASE
    return 0;
}

template <int BN, int BK, int TPS>
static int pool_prepare_cfg()
{
    static bool attr_done[64] = {false};
    int dev = 0;
    Y2_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && !attr_done[dev]) {
        Y2_CUDA_CHECK(cudaFuncSetAttribute(conv_pool_kernel<BN, BK, TPS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           227 * 1024));
        attr_done[dev] = true;
    }
    return Y2_OK;
}

int pool_plan_init(y2_conv_plan *pl, const y2_conv_desc *d)
{
    const int bn = d->npad, bk = d->block_k;
    const int tps = pool_tps(bn, bk);
    if (d->ksize != 3 || d->cin != bk || !tps || d->cout != bn || d->h < 2 || d->w < 2 ||
        (d->act != Y2_ACT_LEAKY && d->act != Y2_ACT_LINEAR)) {
        set_error("conv+pool plan: needs a 3x3 layer with one channel block (cin=%d block_k=%d) and 64 or 128 stored "
                  "filters (cout=%d npad=%d), leaky or linear", d->cin, bk, d->cout, d->npad);
        return Y2_EINVAL;
    }
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) {
        set_error("cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)");
        return Y2_ECUDA;
    }
    const int oh = d->h / 2, ow = d->w / 2;
    // equal, even-width column tiles of at most 126 image columns
    const int nx = (2 * ow + 125) / 126;
    int wt = (2 * ow + nx - 1) / nx;
    wt += wt & 1;
    const int P = wt + 2;
    const int row_bytes = bk * 2;
    const int b_stage = tps * bn * bk * 2;
    const int aux = bn * 8 + 512;
    const int budget = 227 * 1024 - 1024 - aux;
    // rows per patch: as many as leave >= 3 weight stages (halo rows amortise over more output rows)
    int rows = 0, patch_bytes = 0;
    for (int r = 16; r >= 2; r -= 2) {
        const int pb = ((r + 2) * P * row_bytes + 1023) / 1024 * 1024;
        if (budget - kPoolStagesA * pb >= 3 * b_stage && budget - kPoolStagesA * pb >= 4096) {
            rows = r;
            patch_bytes = pb;
            break;
        }
    }
    if (!rows || rows + 2 > 256 || P > 256) {
        set_error("conv+pool plan: patch does not fit shared memory");
        return Y2_EINVAL;
    }
    int stages_b = (budget - kPoolStagesA * patch_bytes) / b_stage;
    if (stages_b > kPoolMaxStagesB) stages_b = kPoolMaxStagesB;
    // A: 3-D box (channels, positions of one image row, rows of the stacked padded images)
    {
        const int hp = d->h + 1, wp = d->w + 1;
        cuuint64_t gdim[3] = {(cuuint64_t)d->cin, (cuuint64_t)wp, (cuuint64_t)hp * d->batch};
        cuuint64_t gstr[2] = {(cuuint64_t)d->in_cs * 2, (cuuint64_t)wp * d->in_cs * 2};
        cuuint32_t box[3] = {(cuuint32_t)bk, (cuuint32_t)P, (cuuint32_t)(rows + 2)};
        cuuint32_t estr[3] = {1, 1, 1};
        CUresult r = enc(&pl->tm_a, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void *>(d->in), gdim, gstr, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, bk == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            set_error("conv+pool plan: cuTensorMapEncodeTiled(A) failed: CUresult %d", (int)r);
            return Y2_ECUDA;
        }
    }
    const int ktot = 9 * d->cin;
    int rc = encode_2d_bf16(&pl->tm_b, d->wt, (uint64_t)ktot, (uint64_t)d->npad, (uint64_t)ktot * 2, (uint32_t)bk,
                            (uint32_t)bn, bk);
    if (rc != Y2_OK) return rc;
    PoolParams &p = pl->pool;
    p.batch = d->batch;
    p.h = d->h;
    p.w = d->w;
    p.oh = oh;
    p.ow = ow;
    p.wt = wt;
    p.rows = rows;
    p.tiles_x = (2 * ow + wt - 1) / wt;
    p.tiles_y = (2 * oh + rows - 1) / rows;
    const long long total = (long long)d->batch * p.tiles_x * p.tiles_y;
    if (total > 0x7fffffffLL) return Y2_EINVAL;
    p.total_tiles = (int)total;
    p.patch_bytes = patch_bytes;
    p.stages_b = stages_b;
    p.act = d->act;
    p.alpha = d->alpha;
    p.beta = d->beta;
    p.out = (__nv_bfloat16 *)d->out;
    p.out_cs = d->out_cs;
    // start with the part of a large input that is still in the L2 (see conv_slab.cu, `reverse`)
    p.reverse = (double)d->batch * (d->h + 1) * (d->w + 1) * d->in_cs * 2.0 > 64e6 && !d->in_order;
    pl->variant = kVariantPool;
    pl->block_n = bn;
    pl->block_k = bk;
    pl->smem_bytes = (size_t)kPoolStagesA * patch_bytes + (size_t)stages_b * b_stage + aux + 1024;
    const int sms = sm_count();
    pl->grid = p.total_tiles < sms ? p.total_tiles : sms;
#define Y2_CASE(BN, BK, TPS) \
    if (bn == BN && bk == BK) return pool_prepare_cfg<BN, BK, TPS>();
    Y2_FOR_EACH_POOL_CFG(Y2_CASE)
#undef Y2_CASE
    return Y2_EINVAL;
}

int pool_plan_launch(const y2_conv_plan *pl, cudaStream_t st)
{
#define Y2_CASE(BN, BK, TPS)                                                                                     \
    if (pl->block_n == BN && pl->block_k == BK) {                                                                \
        Y2_CUDA_CHECK(launch_pdl(conv_pool_kernel<BN, BK, TPS>, dim3(pl->grid), dim3(kPoolThreads), pl->smem_bytes, st, \
                                 pl->tm_a, pl->tm_b, pl->pool));                                                        \
        Y2_LAUNCH_CHECK();                                                                                       \
        return Y2_OK;                                                                                            \
    }
    Y2_FOR_EACH_POOL_CFG(Y2_CASE)
#undef Y2_CASE
    set_error("pool_plan_launch: no kernel for block_n=%d block_k=%d", pl->block_n, pl->block_k);
    return Y2_EINVAL;
}

} // namespace y2
