// Implicit-GEMM convolution for sm_100a: TMA -> smem ring -> tcgen05.mma -> TMEM ->
// fused batchnorm/bias/activation epilogue.
//
// Replaces forward_convolutional_layer_gpu (reference convolutional_kernels.cu:77-131):
//   fill_ongpu + per-image im2col_ongpu + gemm_ongpu(cublasSgemm) + normalize_gpu +
//   scale_bias_gpu + add_bias_gpu + activate_array_ongpu   (2B+6 launches per layer)
// by ONE persistent launch per layer over the whole batch.
//
// GEMM view.  Activations are "padded NHWC" (see yolo2_b200_kernels.h): flat position p,
// CS channels per position, zero pad row/column per image.  For a k x k stride-1 'same'
// convolution
//   D[p][f] = sum_{tap=(r,s)} sum_c  X[p + (r-k/2)*(W+1) + (s-k/2)][c] * Wt[f][(r*k+s)*C + c]
// so the A operand of every tap is the same 2-D tensor (C, P) read at a shifted row
// coordinate; TMA zero-fills rows outside [0, P).  No im2col buffer exists anywhere.
//
// CTA = 6 warps: warp 0 TMA producer, warp 1 MMA issuer (+TMEM alloc), warps 2-5 epilogue.
// Tile = 128 positions x BLOCK_N filters, accumulators double-buffered in TMEM so the
// epilogue of tile i overlaps the MMAs of tile i+1.
#include "conv_plan.cuh"

#include <mutex>
#include <new>
#include <stdlib.h>
#include <string.h>

namespace y2 {

constexpr int kThreads = 192;
constexpr int kMaxStages = 8;

template <int BLOCK_N, int BLOCK_K>
struct ConvCfg {
    static constexpr int kABytes = kBlockM * BLOCK_K * 2;
    static constexpr int kBBytes = BLOCK_N * BLOCK_K * 2;
    static constexpr int kStageBytes = kABytes + kBBytes;
    static constexpr int kTmemCols = (2 * BLOCK_N <= 32) ? 32 : (2 * BLOCK_N <= 64) ? 64
                                   : (2 * BLOCK_N <= 128) ? 128 : (2 * BLOCK_N <= 256) ? 256 : 512;
    // swizzle atom = 8 rows x (BLOCK_K*2) bytes
    static constexpr uint32_t kSBO = 8 * BLOCK_K * 2;
    static constexpr uint32_t kLayout = (BLOCK_K == 64) ? 2u : 4u; // SWIZZLE_128B : SWIZZLE_64B
    // cute::UMMA::InstrDescriptor: c=F32 [4,6), a=BF16 [7,10), b=BF16 [10,13), K-major both,
    // N>>3 at [17,23), M>>4 at [24,29)
    static constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) |
                                       ((uint32_t)(BLOCK_N >> 3) << 17) |
                                       ((uint32_t)(kBlockM >> 4) << 24);
    static constexpr int kAuxBytes = 2 * 2 * BLOCK_N * 4 /*alpha,beta x2*/ + 256 /*barriers*/;
};

template <int BLOCK_N, int BLOCK_K>
__global__ void __launch_bounds__(kThreads, 1)
conv_tcgen05_kernel(const __grid_constant__ CUtensorMap tm_a,
                    const __grid_constant__ CUtensorMap tm_b, const ConvParams prm)
{
    using Cfg = ConvCfg<BLOCK_N, BLOCK_K>;
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment required by the 128B swizzle atoms
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);

    const int stages = prm.stages;
    uint8_t *aux = smem + (size_t)stages * Cfg::kStageBytes;
    float *s_ab = reinterpret_cast<float *>(aux); // [2 acc][alpha BLOCK_N | beta BLOCK_N]
    uint64_t *bars = reinterpret_cast<uint64_t *>(aux + 2 * 2 * BLOCK_N * 4);
    uint64_t *full_bar = bars;
    uint64_t *empty_bar = bars + kMaxStages;
    uint64_t *tfull_bar = bars + 2 * kMaxStages;
    uint64_t *tempty_bar = bars + 2 * kMaxStages + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * kMaxStages + 4);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int total_tiles = prm.tiles_m * prm.tiles_n;
    const int kblocks = prm.taps * prm.cblocks;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tm_a);
        tma_prefetch_desc(&tm_b);
        for (int i = 0; i < stages; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tfull_bar[i], 1);
            mbar_init(&tempty_bar[i], 128);
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
    const uint32_t tmem_base = *tmem_slot;

    pdl_launch_dependents();
    if (warp == 0) {
        // ===================== TMA producer (whole warp waits, one elected lane issues) ==========
        pdl_wait();  // activations = the previous layer's output
        int stage = 0;
        uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const int m_tile = tile / prm.tiles_n;
            const int n_tile = tile - m_tile * prm.tiles_n;
            const int p0 = m_tile * kBlockM;
            const int n0 = n_tile * BLOCK_N;
            int kb = 0;
            for (int tap = 0; tap < prm.taps; ++tap) {
                int shift = 0;
                if (prm.ksize == 3) shift = (tap / 3 - 1) * prm.wp + (tap % 3 - 1);
                for (int cb = 0; cb < prm.cblocks; ++cb, ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1, 1);
                    if (elect_one_sync()) {
                        uint8_t *sa = smem + (size_t)stage * Cfg::kStageBytes;
                        uint8_t *sb = sa + Cfg::kABytes;
                        mbar_expect_tx(&full_bar[stage], Cfg::kStageBytes);
                        tma_load_2d(&tm_a, &full_bar[stage], sa, cb * BLOCK_K, p0 + shift);
                        tma_load_2d(&tm_b, &full_bar[stage], sb, kb * BLOCK_K, n0);
                    }
                    __syncwarp();
                    if (++stage == stages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        int stage = 0;
        uint32_t phase = 0;
        int it = 0;
        uint32_t tok = 0;  // early try_wait on the next stage (its latency overlaps the MMA issue)
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
            const int acc = it & 1;
            const uint32_t acc_phase = (it >> 1) & 1;
            const bool last_tile = tile + (int)gridDim.x >= total_tiles;
            mbar_wait(&tempty_bar[acc], acc_phase ^ 1, 2);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BLOCK_N);
            for (int kb = 0; kb < kblocks; ++kb) {
                if (!tok) mbar_wait(&full_bar[stage], phase, 3);
                tc_fence_after();
                int ns = stage + 1;
                uint32_t np = phase;
                if (ns == stages) { ns = 0; np ^= 1; }
                tok = (last_tile && kb == kblocks - 1) ? 0u : mbar_test_wait(&full_bar[ns], np);
                if (elect_one_sync()) {
                    const uint32_t sa = smem_u32(smem + (size_t)stage * Cfg::kStageBytes);
                    const uint32_t sb = sa + Cfg::kABytes;
                    const uint64_t adesc = make_kmajor_desc(sa, Cfg::kSBO, Cfg::kLayout);
                    const uint64_t bdesc = make_kmajor_desc(sb, Cfg::kSBO, Cfg::kLayout);
#pragma unroll
                    for (int k = 0; k < BLOCK_K / 16; ++k) {
                        // +32 bytes per K=16 step inside the swizzle atom (encoded >>4)
                        umma_bf16(d_tmem, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2),
                                  Cfg::kIdesc, (uint32_t)((kb | k) != 0));
                    }
                    umma_commit(&empty_bar[stage]);
                    if (kb == kblocks - 1) umma_commit(&tfull_bar[acc]);
                }
                __syncwarp();
                stage = ns;
                phase = np;
            }
        }
    } else {
        // ===================== epilogue (warps 2..5) =====================
        const int quarter = warp & 3;            // TMEM lane quarter this warp may read
        const int row = quarter * 32 + lane;     // tile row == TMEM lane
        const int et = threadIdx.x - 64;         // 0..127
        const int img_pos = prm.hp * prm.wp;
        int it = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
            const int acc = it & 1;
            const uint32_t acc_phase = (it >> 1) & 1;
            const int m_tile = tile / prm.tiles_n;
            const int n_tile = tile - m_tile * prm.tiles_n;
            const int n0 = n_tile * BLOCK_N;
            float *sa = s_ab + acc * 2 * BLOCK_N;
            for (int i = et; i < 2 * BLOCK_N; i += 128) {
                sa[i] = (i < BLOCK_N) ? __ldg(prm.alpha + n0 + i) : __ldg(prm.beta + n0 + i - BLOCK_N);
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");

            const int p = m_tile * kBlockM + row;
            const bool in_range = p < prm.total_pos;
            const int b = p / img_pos;
            const int rem = p - b * img_pos;
            const int y = rem / prm.wp;
            const int x = rem - y * prm.wp;
            const bool valid = in_range && (y < prm.h) && (x < prm.w);

            mbar_wait(&tfull_bar[acc], acc_phase, 4);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) +
                                   (uint32_t)(acc * BLOCK_N);
#pragma unroll 1
            for (int c0 = 0; c0 < BLOCK_N; c0 += 32) {
                uint32_t v[32];
                tmem_ld32(taddr + (uint32_t)c0, v);
                tmem_ld_wait();
                float f[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    float t = fmaf(__uint_as_float(v[j]), sa[c0 + j], sa[BLOCK_N + c0 + j]);
                    if (prm.act == Y2_ACT_LEAKY) t = (t > 0.f) ? t : 0.1f * t;
                    else if (prm.act == Y2_ACT_LOGISTIC) t = 1.f / (1.f + __expf(-t));
                    f[j] = t;
                }
                const int ch0 = n0 + c0;
                if (prm.out_mode == Y2_OUT_BF16_PADDED) {
                    if (in_range) {
                        __nv_bfloat16 *o = reinterpret_cast<__nv_bfloat16 *>(prm.out) +
                                           (size_t)p * prm.out_cs + ch0;
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
                } else { // Y2_OUT_F32_FLAT: [B][h*w][out_cs]
                    if (valid) {
                        float *o = reinterpret_cast<float *>(prm.out) +
                                   ((size_t)b * prm.h * prm.w + (size_t)y * prm.w + x) * prm.out_cs +
                                   ch0;
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (ch0 + j < prm.cout) o[j] = f[j];
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(&tempty_bar[acc]);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                     "r"((uint32_t)Cfg::kTmemCols)
                     : "memory");
    }
}

// -------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------
EncodeTiledFn get_encode_fn()
{
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
        if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = (EncodeTiledFn)p;
    });
    return fn;
}

int encode_2d_bf16(CUtensorMap *tm, const void *base, uint64_t dim0, uint64_t dim1,
                          uint64_t stride1_bytes, uint32_t box0, uint32_t box1, int block_k)
{
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) {
        set_error("cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)");
        return Y2_ECUDA;
    }
    cuuint64_t gdim[2] = {dim0, dim1};
    cuuint64_t gstr[1] = {stride1_bytes};
    cuuint32_t box[2] = {box0, box1};
    cuuint32_t estr[2] = {1, 1};
    CUtensorMapSwizzle sw = (block_k == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(base), gdim, gstr,
                    box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed: CUresult %d (dims %llu x %llu, stride %llu, box %u x %u)",
                  (int)r, (unsigned long long)dim0, (unsigned long long)dim1,
                  (unsigned long long)stride1_bytes, box0, box1);
        return Y2_ECUDA;
    }
    return Y2_OK;
}

} // namespace y2

namespace y2 {

template <int BN, int BK>
static int prepare_cfg()
{
    // raise the dynamic shared-memory limit once per device; done at plan time so that nothing
    // but the launch itself happens inside a CUDA-graph capture
    static bool attr_done[64] = {false};
    int dev = 0;
    Y2_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && !attr_done[dev]) {
        Y2_CUDA_CHECK(cudaFuncSetAttribute(conv_tcgen05_kernel<BN, BK>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        attr_done[dev] = true;
    }
    return Y2_OK;
}

template <int BN, int BK>
static int launch_cfg(const y2_conv_plan *pl, cudaStream_t st)
{
    Y2_CUDA_CHECK(launch_pdl(conv_tcgen05_kernel<BN, BK>, dim3(pl->grid), dim3(kThreads), pl->smem_bytes, st, pl->tm_a,
                             pl->tm_b, pl->prm));
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

#define Y2_FOR_EACH_CFG(X) X(256, 64) X(128, 64) X(64, 64) X(32, 64) X(128, 32) X(64, 32) X(32, 32)

static int prepare(int block_n, int block_k)
{
#define Y2_CASE(BN, BK) \
    if (block_n == BN && block_k == BK) return prepare_cfg<BN, BK>();
    Y2_FOR_EACH_CFG(Y2_CASE)
#undef Y2_CASE
    set_error("no conv kernel for block_n=%d block_k=%d", block_n, block_k);
    return Y2_EINVAL;
}

} // namespace y2

extern "C" int y2_conv_plan_create(const y2_conv_desc *d, y2_conv_plan **out_plan)
{
    using namespace y2;
    if (!d || !out_plan) return Y2_EINVAL;
    *out_plan = nullptr;
    const bool bn_ok = d->block_n == 32 || d->block_n == 64 || d->block_n == 128 || d->block_n == 256;
    const bool bk_ok = d->block_k == 64 || d->block_k == 32;
    if (!bn_ok || !bk_ok || (d->ksize != 1 && d->ksize != 3) || d->cin <= 0 || d->cin % d->block_k ||
        d->npad <= 0 || d->npad % d->block_n || d->in_cs % 8 || d->batch <= 0 || d->h <= 0 || d->w <= 0 ||
        d->cout <= 0 || d->cout > d->npad || !d->in || !d->wt || !d->out || !d->alpha || !d->beta) {
        set_error("y2_conv_plan_create: invalid descriptor (block_n=%d block_k=%d ksize=%d cin=%d npad=%d "
                  "in_cs=%d cout=%d)", d->block_n, d->block_k, d->ksize, d->cin, d->npad, d->in_cs, d->cout);
        return Y2_EINVAL;
    }
    if (d->out_mode != Y2_OUT_F32_FLAT && (d->out_cs % 8 || d->cout % 8 ||
                                              ((uintptr_t)d->out & 15))) {
        set_error("y2_conv_plan_create: bf16 output needs 16-byte aligned channel slices");
        return Y2_EINVAL;
    }
    if (((uintptr_t)d->in & 15) || ((uintptr_t)d->wt & 15)) {
        set_error("y2_conv_plan_create: operands must be 16-byte aligned");
        return Y2_EINVAL;
    }
    y2_conv_plan *pl = new (std::nothrow) y2_conv_plan();
    if (!pl) return Y2_ENOMEM;
    const int hp = d->h + 1, wp = d->w + 1;
    const long long total = (long long)d->batch * hp * wp;
    if (total > 0x7fffff00LL) {
        delete pl;
        set_error("y2_conv_plan_create: too many positions");
        return Y2_EINVAL;
    }
    const int taps = d->ksize * d->ksize;
    const int ktot = taps * d->cin;
    // kernel choice: CTA-pair kernel for wide 3x3 layers, halo-slab kernel for the other 3x3 layers, this
    // file's per-tap kernel for 1x1 layers and whatever does not fit.  Y2_CONV_VARIANT=pertap|slab|pair
    // restricts the choice (tests, A/B timing); slab and pair also lift the slab kernel's 1x1 preference, pair
    // admits 1x1 layers to the one-tap pair kernel.
    if (d->out_mode == Y2_OUT_BF16_POOLED) {
        const int rc = pool_plan_init(pl, d);
        if (rc != Y2_OK) {
            delete pl;
            return rc;
        }
        *out_plan = pl;
        return Y2_OK;
    }
    const char *forced = getenv("Y2_CONV_VARIANT");
    const ConvChoice choice = !forced                  ? kChooseAuto
                              : !strcmp(forced, "slab") ? kChooseSlab
                              : !strcmp(forced, "pair") ? kChoosePair
                                                        : kChoosePerTap;
    if ((choice == kChooseAuto || choice == kChoosePair) && pair_plan_init(pl, d, choice) == Y2_OK) {
        *out_plan = pl;
        return Y2_OK;
    }
    if (choice != kChoosePerTap && slab_plan_init(pl, d, choice) == Y2_OK) {
        *out_plan = pl;
        return Y2_OK;
    }
    pl->variant = kVariantPerTap;
    int rc = encode_2d_bf16(&pl->tm_a, d->in, (uint64_t)d->cin, (uint64_t)total, (uint64_t)d->in_cs * 2,
                            (uint32_t)d->block_k, kBlockM, d->block_k);
    if (rc == Y2_OK)
        rc = encode_2d_bf16(&pl->tm_b, d->wt, (uint64_t)ktot, (uint64_t)d->npad, (uint64_t)ktot * 2,
                            (uint32_t)d->block_k, (uint32_t)d->block_n, d->block_k);
    if (rc != Y2_OK) {
        delete pl;
        return rc;
    }
    ConvParams &p = pl->prm;
    p.taps = taps;
    p.ksize = d->ksize;
    p.cblocks = d->cin / d->block_k;
    p.wp = wp;
    p.hp = hp;
    p.h = d->h;
    p.w = d->w;
    p.total_pos = (int)total;
    p.tiles_m = (int)((total + kBlockM - 1) / kBlockM);
    p.tiles_n = d->npad / d->block_n;
    p.cout = d->cout;
    p.act = d->act;
    p.out_mode = d->out_mode;
    p.out_cs = d->out_cs;
    p.alpha = d->alpha;
    p.beta = d->beta;
    p.out = d->out;
    pl->block_n = d->block_n;
    pl->block_k = d->block_k;
    const int stage_bytes = (kBlockM + d->block_n) * d->block_k * 2;
    const int aux = 2 * 2 * d->block_n * 4 + 256;
    int stages = (227 * 1024 - 1024 - aux) / stage_bytes;
    if (stages > kMaxStages) stages = kMaxStages;
    if (stages < 2) {
        delete pl;
        set_error("y2_conv_plan_create: tile does not fit shared memory");
        return Y2_EINVAL;
    }
    p.stages = stages;
    pl->smem_bytes = (size_t)stages * stage_bytes + aux + 1024;
    const int tiles = p.tiles_m * p.tiles_n;
    const int sms = sm_count();
    pl->grid = tiles < sms ? tiles : sms;
    rc = prepare(d->block_n, d->block_k);
    if (rc != Y2_OK) {
        delete pl;
        return rc;
    }
    *out_plan = pl;
    return Y2_OK;
}

extern "C" int y2_conv_plan_launch(const y2_conv_plan *pl, y2_stream_t s)
{
    using namespace y2;
    if (!pl) return Y2_EINVAL;
    cudaStream_t st = to_stream(s);
    if (pl->variant == kVariantPool) return pool_plan_launch(pl, st);
    if (pl->variant == kVariantPair) return pair_plan_launch(pl, st);
    if (pl->variant == kVariantSlab) return slab_plan_launch(pl, st);
#define Y2_CASE(BN, BK) \
    if (pl->block_n == BN && pl->block_k == BK) return launch_cfg<BN, BK>(pl, st);
    Y2_FOR_EACH_CFG(Y2_CASE)
#undef Y2_CASE
    set_error("y2_conv_plan_launch: no kernel for block_n=%d block_k=%d", pl->block_n, pl->block_k);
    return Y2_EINVAL;
}

extern "C" void y2_conv_plan_destroy(y2_conv_plan *pl)
{
    if (!pl) return;
    if (pl->work_buf) cudaFree(pl->work_buf);
    delete pl;
}

extern "C" int y2_conv_plan_order(const y2_conv_plan *pl)
{
    if (!pl) return 0;
    if (pl->variant == y2::kVariantSlab) return pl->slab.reverse;
    if (pl->variant == y2::kVariantPool) return pl->pool.reverse;
    return 0;
}

extern "C" int y2_conv_plan_variant(const y2_conv_plan *pl)
{
    return pl ? pl->variant : -1;
}

extern "C" int y2_conv_plan_tiles(const y2_conv_plan *pl)
{
    if (!pl) return 0;
    if (pl->variant == y2::kVariantPool) return pl->pool.total_tiles;
    return pl->variant != y2::kVariantPerTap ? pl->slab.tiles_m * pl->slab.tiles_n : pl->prm.tiles_m * pl->prm.tiles_n;
}
