// Shared definition of a convolution plan: tensor maps + launch geometry of one of the two
// tcgen05 implicit-GEMM kernels (conv_slab.cu: halo slab + dual accumulators; conv_tcgen05.cu:
// one TMA load per tap, the general fallback).
#pragma once
#include "y2_common.cuh"

namespace y2 {

constexpr int kBlockM = 128;

// ---- per-tap kernel (conv_tcgen05.cu) ------------------------------------------------
struct ConvParams {
    int taps;        // 1 or 9
    int ksize;       // 1 or 3
    int cblocks;     // cin / BLOCK_K
    int wp, hp;      // padded row pitch / rows per image
    int h, w;
    int total_pos;   // B * hp * wp
    int tiles_m, tiles_n;
    int cout;        // channels stored
    int act;
    int out_mode;
    int out_cs;
    int stages;
    const float *alpha;
    const float *beta;
    void *out;
};

// ---- slab kernel (conv_slab.cu) ------------------------------------------------------
// The slab and pair kernels take it __grid_constant__, so its fields are read from the parameter bank where they
// are used.  Without the qualifier the 128-byte struct is copied into registers up front, and the CTA-pair 3x3
// kernel spills more.
struct SlabParams {
    int cblocks;           // cin / BLOCK_K
    int wp, hp, h, w;
    int total_pos;
    int tiles_m, tiles_n;  // tiles_m counts tiles of ACCS x 128 positions
    int halo;              // rows of the slab before the tile's first position (wp + 1)
    int slab_loads;        // TMA loads per slab
    int box_rows;          // rows per TMA load
    int slab_bytes;        // bytes per slab stage
    int stages_a, stages_b;
    int cout, act, out_mode, out_cs;
    int tma_store;         // bf16 output leaves through per-warp TMA stores (else direct 16-byte stores)
    int couple;            // epilogue warps re-synchronise every tile even when (alpha, beta) do not change
    int reverse;           // slab kernel: walk the position tiles last-to-first (see slab_plan_init)
    const int4 *work;      // pair kernel: per-pair lists of pieces (m_tile, n0, ncols, -), ncols == 0 terminates
    int work_stride;       // entries per pair in `work`
    const float *alpha;
    const float *beta;
    void *out;
};

// ---- conv + 2x2 maxpool kernel (conv_pool.cu) ------------------------------------------
struct PoolParams {
    int batch, h, w;       // conv extent (stride-1 'same': input == output extent)
    int oh, ow;            // pooled extent
    int wt;                // image columns per tile (even); patch row = wt + 2 positions
    int rows;              // image rows per patch (even)
    int tiles_x, tiles_y, total_tiles;
    int patch_bytes;       // bytes per patch stage (multiple of 1024)
    int stages_b;
    int act;
    const float *alpha;
    const float *beta;
    __nv_bfloat16 *out;    // pooled padded NHWC [B][oh+1][ow+1][out_cs]
    int out_cs;
    int reverse;           // walk the tiles last-to-first (input near / above the L2 capacity, see conv_slab.cu)
};

enum { kVariantPerTap = 0, kVariantSlab = 1, kVariantPair = 2, kVariantPool = 3 };

// Y2_CONV_VARIANT, read once per plan by y2_conv_plan_create: unset = auto, pertap | slab | pair restrict the
// choice (an unknown value is pertap)
enum ConvChoice { kChooseAuto, kChoosePerTap, kChooseSlab, kChoosePair };

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *,
                                  const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode_fn();
// 2-D bf16 tensor map (dim0 = channels, contiguous; dim1 = rows), swizzle = box0 bytes
int encode_2d_bf16(CUtensorMap *tm, const void *base, uint64_t dim0, uint64_t dim1,
                   uint64_t stride1_bytes, uint32_t box0, uint32_t box1, int block_k);

} // namespace y2

struct y2_conv_plan {
    CUtensorMap tm_a;
    CUtensorMap tm_b;
    CUtensorMap tm_out;  // slab kernel: the output tensor (TMA stores)
    CUtensorMap tm_b32;  // pair kernel: the weights in 32-filter boxes (narrow pieces)
    int variant;
    y2::ConvParams prm;
    y2::SlabParams slab;
    y2::PoolParams pool;
    int block_n, block_k, taps;
    int grid;
    size_t smem_bytes;
    void *work_buf = nullptr;  // device copy of the pair kernel's work lists, owned by the plan
};

namespace y2 {
// conv_slab.cu: returns Y2_OK and fills the plan when the layer fits the slab kernel, Y2_EINVAL
// (without touching the error string) when it does not and the per-tap kernel must be used
int slab_plan_init(y2_conv_plan *pl, const y2_conv_desc *d, ConvChoice choice);
int slab_plan_launch(const y2_conv_plan *pl, cudaStream_t st);
// conv_pair.cu: the CTA-pair (cta_group::2) kernel for wide 3x3 layers, same contract
int pair_plan_init(y2_conv_plan *pl, const y2_conv_desc *d, ConvChoice choice);
int pair_plan_launch(const y2_conv_plan *pl, cudaStream_t st);
// conv_pool.cu: 3x3 convolution fused with the following 2x2/2 maxpool (out_mode Y2_OUT_BF16_POOLED)
int pool_plan_init(y2_conv_plan *pl, const y2_conv_desc *d);
int pool_plan_launch(const y2_conv_plan *pl, cudaStream_t st);
} // namespace y2
