// Implicit-GEMM 3x3 convolution on CTA pairs: tcgen05.mma.cta_group::2 over a 2-CTA cluster.
//
// Replaces forward_convolutional_layer_gpu (reference convolutional_kernels.cu:77-131) for the wide
// 3x3 layers (>= 256 filters, C_in a multiple of 64) - two thirds of YOLOv2's FLOPs.
//
// Why pairs.  With one CTA per tile (conv_slab.cu) a 128 x 256 x 64 MMA step moves 34 KB into shared
// memory and reads 48 KB of operands back out of it in 512 tensor-pipe clocks: the ~128 B/clk/SM of
// shared-memory bandwidth, not the tensor pipe, bounds the layer at ~60% of peak.  A CTA pair
// computes a 256 x 256 tile with ONE instruction stream: each CTA holds its own 128 positions of the
// halo slab (A) and HALF of the 256-filter weight tile (B); the tensor cores of both SMs read the
// two halves across the pair.  Per SM and step that is 18 KB of fill and 32 KB of operand reads.
//
// Protocol (leader = even CTA of the pair):
//   * both CTAs TMA-load their slab / weight half into their own shared memory; the bytes are
//     credited to the LEADER's full barriers (.cta_group::2 TMA, peer bit cleared in the mbarrier
//     address), whose single arrival is the leader's expect_tx for both halves;
//   * only the leader issues MMAs; tcgen05.commit multicasts the "stage free" / "accumulator
//     full" arrivals to the barriers at the same offset in both CTAs;
//   * each CTA drains its own 128 TMEM lanes; "accumulator drained" arrivals of both CTAs land on
//     the leader's barrier (remote mbarrier.arrive through mapa).
// Everything else (halo slab, row-shifted descriptors, double-buffered accumulators, 8 epilogue
// warps) is conv_slab.cu's design.
//
// Work distribution.  Whole 256 x 256 tiles round-robin leave the last wave partly empty when the tile count is
// a small non-multiple of the 74 pairs (13x13 layers at batch 64: 196 tiles = 2.65 waves, run as 3).  The host
// therefore hands every pair an explicit list of PIECES (position tile, first filter, 64..256 filters): the
// (position tile, 64-filter unit) sequence is cut into one contiguous range per pair such that the largest range
// cost is minimal under a measured cost model of narrow pieces, and every range is split into pieces of at most
// 256 filters.  A piece is a full K loop over N = 64..256 filters (tcgen05.mma N is a runtime field of the
// instruction descriptor), so every output element is still accumulated by ONE pair in the same order: results
// are bit-identical to whole tiles, nothing is parked or joined (the stream-K schedule this replaces needed fp32
// partial sums in global scratch and lost at the power cap, DESIGN.md 3.3).  Y2_PAIR_BALANCE=0 restores whole
// tiles round-robin (same kernel, different list).
//
// One-tap form (TAPS = 1, 1x1 layers).  Used by default only for wide fp32 heads (yolo9000's 28 269 filters over 1024
// channels: 1263 -> 985 us at batch 64 against the single-CTA slab kernel, whose 128 x 256 MMAs are operand-fetch
// bound); for the bf16 1x1 layers of the detectors it measured no faster than the slab kernel and is opt-in
// (pair_plan_init).
#include "conv_epilogue.cuh"

#include <stdlib.h>
#include <string.h>

#include <vector>

namespace y2 {

constexpr int kPairThreads = 352;
constexpr int kPairEpiThreads = 256;
constexpr int kPairMaxStagesA = 4;
constexpr int kPairMaxStagesB = 10;
constexpr int kPairBK = 64;
constexpr int kPairN = 256;                          // filters per pair tile
constexpr int kPairRowBytes = kPairBK * 2;           // 128
constexpr int kPairBHalfBytes = 128 * kPairBK * 2;   // this CTA's half of a weight tile
constexpr uint32_t kPairDescHi = ((8u * kPairRowBytes) >> 4) | (1u << 14) | (2u << 29);  // SBO 1024, v1, SWIZZLE_128B
// c = F32, a = b = BF16, K-major, M = 256 (both CTAs); N (64 ... 256) is or-ed in per piece at bit 17
constexpr uint32_t kPairIdescM = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(256 >> 4) << 24);

// one piece of work: a full K loop over `ncols` filters (64, 128, 192 or 256) of one position tile
struct PairSeg {
    int m_tile, n0, ncols;
};

// this pair's list: int4 (m_tile, n0, ncols, -) entries, ncols == 0 terminates
struct PairSched {
    const int4 *w;
    __device__ PairSched(const SlabParams &prm, int pair) : w(prm.work + (size_t)pair * prm.work_stride) {}
    __device__ bool next(PairSeg &s)
    {
        if (!peek(s)) return false;
        ++w;
        return true;
    }
    __device__ bool peek(PairSeg &s) const
    {
        const int4 q = __ldg(w);
        s.m_tile = q.x;
        s.n0 = q.y;
        s.ncols = q.z;
        return q.z != 0;
    }
};

// TAPS = 9: 3x3 layer (halo slab, nine row-shifted descriptors per channel block);
// TAPS = 1: 1x1 layer (the "slab" is the plain 128-position tile, one descriptor per channel block)
template <int TAPS>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kPairThreads, 1)
conv_pair_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                 const __grid_constant__ CUtensorMap tm_b32, const __grid_constant__ CUtensorMap tm_out,
                 const __grid_constant__ SlabParams prm)
{
    extern __shared__ uint8_t smem_raw[];
    // identical carve-up in both CTAs: descriptors and barrier offsets name the peer's memory too
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);

    const int stages_a = prm.stages_a, stages_b = prm.stages_b;
    uint8_t *smem_a = smem;
    uint8_t *smem_b = smem + (size_t)stages_a * prm.slab_bytes;
    uint8_t *aux = smem_b + (size_t)stages_b * kPairBHalfBytes;
    float2 *s_ab = reinterpret_cast<float2 *>(aux);  // [2 buf][256] (alpha, beta)
    uint64_t *bars = reinterpret_cast<uint64_t *>(aux + 2 * kPairN * 8);
    uint64_t *a_full = bars;
    uint64_t *a_empty = bars + kPairMaxStagesA;
    uint64_t *b_full = bars + 2 * kPairMaxStagesA;
    uint64_t *b_empty = b_full + kPairMaxStagesB;
    uint64_t *tfull_bar = b_empty + kPairMaxStagesB;
    uint64_t *tempty_bar = tfull_bar + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty_bar + 2);
    // [8 epilogue warps][32 rows][128 B] staging of the TMA stores, 1024-byte aligned (swizzle atom)
    uint4 *s_stage = reinterpret_cast<uint4 *>(aux + ((2 * kPairN * 8 + 512 + 1023) / 1024) * 1024);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int pair = blockIdx.x >> 1;
    const int cblocks = prm.cblocks;
    PairSched sched(prm, pair);
    PairSeg seg;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tm_a);
        tma_prefetch_desc(&tm_b);
        tma_prefetch_desc(&tm_b32);
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
            mbar_init(&tempty_bar[i], 2 * kPairEpiThreads);  // the epilogue threads of both CTAs
        }
        fence_barrier_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    cluster_sync_all();  // barriers of both CTAs initialised before any remote arrival
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    pdl_launch_dependents();
    if (warp == 0) {
        // ===================== slab producer (both CTAs, own 128 positions) =====================
        pdl_wait();  // the activations are the previous layer's output; weights (warp 2) are prefetched meanwhile
        int stage = 0;
        uint32_t phase = 0;
        const uint32_t slab_tx = (uint32_t)prm.slab_loads * prm.box_rows * kPairRowBytes;
        const uint32_t load_bytes = (uint32_t)prm.box_rows * kPairRowBytes;
        while (sched.next(seg)) {
            const int row0 = seg.m_tile * 256 + (int)rank * 128 - prm.halo;
            for (int cb = 0; cb < cblocks; ++cb) {
                mbar_wait(&a_empty[stage], phase ^ 1, 1);
                if (elect_one_sync()) {
                    uint8_t *sa = smem_a + (size_t)stage * prm.slab_bytes;
                    if (leader) mbar_expect_tx(&a_full[stage], 2 * slab_tx);
                    for (int i = 0; i < prm.slab_loads; ++i)
                        tma_load_2d_pair(&tm_a, &a_full[stage], sa + i * load_bytes, cb * kPairBK,
                                         row0 + i * prm.box_rows);
                }
                __syncwarp();
                if (++stage == stages_a) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 2) {
        // ===================== weight producer (both CTAs, own half of the piece's filters) =====
        int stage = 0;
        uint32_t phase = 0;
        while (sched.next(seg)) {
            const int half_rows = seg.ncols >> 1;  // 32, 64, 96 or 128 filters per CTA
            const int n0 = seg.n0 + (int)rank * half_rows;
            const uint32_t tx = (uint32_t)seg.ncols * kPairRowBytes;  // both halves
            for (int cb = 0; cb < cblocks; ++cb) {
#pragma unroll 1
                for (int tap = 0; tap < TAPS; ++tap) {
                    mbar_wait(&b_empty[stage], phase ^ 1, 2);
                    if (elect_one_sync()) {
                        uint8_t *sb = smem_b + (size_t)stage * kPairBHalfBytes;
                        const int k0 = (tap * cblocks + cb) * kPairBK;
                        if (leader) mbar_expect_tx(&b_full[stage], tx);
                        if (half_rows == 128) {
                            tma_load_2d_pair(&tm_b, &b_full[stage], sb, k0, n0);
                        } else {  // narrow piece: 32-filter boxes, only the rows the MMA reads
                            for (int r = 0; r < half_rows; r += 32)
                                tma_load_2d_pair(&tm_b32, &b_full[stage], sb + r * kPairRowBytes, k0, n0 + r);
                        }
                    }
                    __syncwarp();
                    if (++stage == stages_b) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (leader CTA only) =====================
        if (leader) {
            int sa_i = 0, sb_i = 0;
            uint32_t pa = 0, pb = 0;
            int it = 0;
            const uint32_t a_lo0 = ((smem_u32(smem_a) & 0x3FFFFu) >> 4) | (1u << 16);
            const uint32_t b_lo0 = ((smem_u32(smem_b) & 0x3FFFFu) >> 4) | (1u << 16);
            const uint32_t slab16 = (uint32_t)prm.slab_bytes >> 4;
            constexpr uint32_t kRow16 = kPairRowBytes >> 4;
            const uint32_t wp16 = (uint32_t)prm.wp * kRow16;
            for (; sched.next(seg); ++it) {
                const int buf = it & 1;
                const uint32_t buf_phase = (it >> 1) & 1;
                mbar_wait(&tempty_bar[buf], buf_phase ^ 1, 3);
                tc_fence_after();
                const uint32_t d0 = tmem_base + (uint32_t)(buf * kPairN);
                const uint32_t idesc = kPairIdescM | ((uint32_t)(seg.ncols >> 3) << 17);
                for (int cb = 0; cb < cblocks; ++cb) {
                    mbar_wait(&a_full[sa_i], pa, 4);
                    const uint32_t a_lo = a_lo0 + (uint32_t)sa_i * slab16;
                    const uint32_t acc_first = cb != 0;
#pragma unroll
                    for (int tap = 0; tap < TAPS; ++tap) {
                        mbar_wait(&b_full[sb_i], pb, 5);
                        tc_fence_after();
                        if (elect_one_sync()) {
                            const uint32_t b_lo = b_lo0 + (uint32_t)sb_i * (kPairBHalfBytes >> 4);
                            const uint32_t a_tap = a_lo + (uint32_t)(tap / 3) * wp16 + (uint32_t)(tap % 3) * kRow16;
#pragma unroll
                            for (int k = 0; k < kPairBK / 16; ++k)
                                umma_bf16_pair(d0, ((uint64_t)kPairDescHi << 32) | (uint64_t)(a_tap + (uint32_t)(k * 2)),
                                               ((uint64_t)kPairDescHi << 32) | (uint64_t)(b_lo + (uint32_t)(k * 2)),
                                               idesc, (tap == 0 && k == 0) ? acc_first : 1u);
                            umma_commit_pair(&b_empty[sb_i]);
                            if (tap == TAPS - 1) {
                                umma_commit_pair(&a_empty[sa_i]);
                                if (cb == cblocks - 1) umma_commit_pair(&tfull_bar[buf]);
                            }
                        }
                        __syncwarp();
                        if (++sb_i == stages_b) { sb_i = 0; pb ^= 1; }
                    }
                    if (++sa_i == stages_a) { sa_i = 0; pa ^= 1; }
                }
            }
        }
    } else {
        // ===================== epilogue (warps 3..10 of both CTAs, own 128 TMEM lanes) ==========
        // 64-column chunks of the piece alternate between the two warp groups (warps 3-6: chunks 0, 2; warps
        // 7-10: chunks 1, 3)
        const int quarter = warp & 3;
        const int half = (warp - 3) >> 2;
        const int et = threadIdx.x - 96;  // 0..255
        const int img_pos = prm.hp * prm.wp;
        int it = 0;
        if (sched.peek(seg) && et < seg.ncols)
            s_ab[et] = make_float2(__ldg(prm.alpha + seg.n0 + et), __ldg(prm.beta + seg.n0 + et));
        for (; sched.next(seg); ++it) {
            const int buf = it & 1;
            const uint32_t buf_phase = (it >> 1) & 1;
            const int n0 = seg.n0;
            const int nchunks = seg.ncols >> 6;
            const float2 *sab = s_ab + buf * kPairN;
            asm volatile("bar.sync 1, 256;" ::: "memory");  // sab[buf] written, sab[buf ^ 1] free
            PairSeg nseg;
            const bool has_next = sched.peek(nseg);
            float2 ab_next = make_float2(1.f, 0.f);
            if (has_next && et < nseg.ncols)
                ab_next = make_float2(__ldg(prm.alpha + nseg.n0 + et), __ldg(prm.beta + nseg.n0 + et));
            const int p = seg.m_tile * 256 + (int)rank * 128 + quarter * 32 + lane;
            const bool in_range = p < prm.total_pos;
            const int b = p / img_pos;
            const int rem = p - b * img_pos;
            const int y = rem / prm.wp;
            const int x = rem - y * prm.wp;
            const bool valid = in_range && (y < prm.h) && (x < prm.w);
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(buf * kPairN);

            mbar_wait(&tfull_bar[buf], buf_phase, 6);
            tc_fence_after();
            if (half >= nchunks) {  // a 64-filter piece: nothing for the second group to drain
                tc_fence_before();
                mbar_arrive_cluster(&tempty_bar[buf], 0);
            }
#pragma unroll 1
            for (int ch = half; ch < nchunks; ch += 2) {
                const int c = ch * 64;
                uint32_t v0[32], v1[32];
                tmem_ld32(taddr + (uint32_t)c, v0);
                tmem_ld32(taddr + (uint32_t)(c + 32), v1);
                tmem_ld_wait();
                if (ch + 2 >= nchunks) {  // this group's part is in registers: hand it back to the leader's MMA warp
                    tc_fence_before();
                    mbar_arrive_cluster(&tempty_bar[buf], 0);
                }
                if (prm.tma_store == 2) {  // fp32 flat head: staged, row-contiguous 16-byte stores
                    const long long fr = valid ? ((long long)b * prm.h + y) * prm.w + x : -1ll;
                    uint4 *st = s_stage + (warp - 3) * 256;
                    if (prm.act == Y2_ACT_LINEAR) {
                        slab_store_f32_staged<Y2_ACT_LINEAR>(prm, st, v0, sab, c, n0, fr, lane);
                        slab_store_f32_staged<Y2_ACT_LINEAR>(prm, st, v1, sab, c + 32, n0, fr, lane);
                    } else if (prm.act == Y2_ACT_LEAKY) {
                        slab_store_f32_staged<Y2_ACT_LEAKY>(prm, st, v0, sab, c, n0, fr, lane);
                        slab_store_f32_staged<Y2_ACT_LEAKY>(prm, st, v1, sab, c + 32, n0, fr, lane);
                    } else {
                        slab_store_f32_staged<Y2_ACT_LOGISTIC>(prm, st, v0, sab, c, n0, fr, lane);
                        slab_store_f32_staged<Y2_ACT_LOGISTIC>(prm, st, v1, sab, c + 32, n0, fr, lane);
                    }
                } else if (prm.tma_store) {  // bf16 tensor: staged, one TMA store per warp and 64 channels
                    uint4 w[8];
                    if (prm.act == Y2_ACT_LEAKY) {
                        slab_affine_pack<Y2_ACT_LEAKY>(v0, sab, c, valid, w);
                        slab_affine_pack<Y2_ACT_LEAKY>(v1, sab, c + 32, valid, w + 4);
                    } else if (prm.act == Y2_ACT_LINEAR) {
                        slab_affine_pack<Y2_ACT_LINEAR>(v0, sab, c, valid, w);
                        slab_affine_pack<Y2_ACT_LINEAR>(v1, sab, c + 32, valid, w + 4);
                    } else {
                        slab_affine_pack<Y2_ACT_LOGISTIC>(v0, sab, c, valid, w);
                        slab_affine_pack<Y2_ACT_LOGISTIC>(v1, sab, c + 32, valid, w + 4);
                    }
                    slab_store_tma(&tm_out, s_stage + (warp - 3) * 256, w, lane, p - lane, n0 + c);
                } else if (prm.act == Y2_ACT_LEAKY) {
                    slab_epilogue_chunk<Y2_ACT_LEAKY>(prm, v0, sab, c, n0, p, b, y, x, in_range, valid);
                    slab_epilogue_chunk<Y2_ACT_LEAKY>(prm, v1, sab, c + 32, n0, p, b, y, x, in_range, valid);
                } else if (prm.act == Y2_ACT_LINEAR) {
                    slab_epilogue_chunk<Y2_ACT_LINEAR>(prm, v0, sab, c, n0, p, b, y, x, in_range, valid);
                    slab_epilogue_chunk<Y2_ACT_LINEAR>(prm, v1, sab, c + 32, n0, p, b, y, x, in_range, valid);
                } else {
                    slab_epilogue_chunk<Y2_ACT_LOGISTIC>(prm, v0, sab, c, n0, p, b, y, x, in_range, valid);
                    slab_epilogue_chunk<Y2_ACT_LOGISTIC>(prm, v1, sab, c + 32, n0, p, b, y, x, in_range, valid);
                }
            }
            if (has_next) s_ab[(buf ^ 1) * kPairN + et] = ab_next;
        }
        if (prm.tma_store == 1 && lane == 0) tma_store_wait_all();  // the copies read this CTA's shared memory
    }

    tc_fence_before();
    cluster_sync_all();  // no CTA leaves while its peer may still address its shared memory / barriers
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// -------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------
// ---- work lists ------------------------------------------------------------------------
// Cost of one piece of n 64-filter units, in units of a quarter of a full 256-filter piece.  Measured on B200
// (yolo-voc L23 at batch 64 with every piece forced to one width, profiles/r2k_pair_balance.txt; the switch that
// forced the width was removed later and is in the history):
// a tcgen05.mma.cta_group::2 of M = 256, K = 16 takes ~95 / 105 / 115 / 128 clk at N = 64 / 128 / 192 / 256, i.e. it
// has a floor of ~90 clk whatever N is - each SM fetches its 4 KB A operand (and N/2 rows of B) from shared memory at
// ~64 B/clk, which at N = 256 (8 KB) is exactly the 128 clk the tensor pipe needs.  Narrow pieces are therefore
// expensive and the balanced cut only uses them where they shorten the longest list (the 13x13 layers: -1.3 %).
static constexpr double kPairPieceCost[5] = {0.0, 2.97, 3.28, 3.6, 4.0};

// rows = position tiles, U = 64-filter units per row (a multiple of 4), P pairs.
// balanced: the row-major unit sequence is cut into P contiguous ranges of minimal largest cost (binary search on
// the bound, greedy longest-range check - exact for contiguous partitions with a monotone range cost); the units a
// range owns in one row are split into the cheapest pieces of <= 4 units.  Otherwise whole 4-unit pieces round-robin.
static void pair_schedule(int rows, int U, int P, bool balanced, std::vector<int4> &work, int &stride)
{
    std::vector<std::vector<int4>> lists(P);
    const long long T = (long long)rows * U;
    if (balanced && rows * (U / 4) > P) {
        const double *c = kPairPieceCost;
        std::vector<double> g(U + 1, 0.0);   // cheapest split of r units of one row
        std::vector<int> first(U + 1, 0);    // size of the first piece of that split
        for (int r = 1; r <= U; ++r) {
            g[r] = 1e30;
            for (int n = 1; n <= 4 && n <= r; ++n)
                if (c[n] + g[r - n] < g[r] - 1e-9) { g[r] = c[n] + g[r - n]; first[r] = n; }
        }
        std::vector<double> gm(g);  // monotone envelope: owning fewer units of a row never counts as more
        for (int r = U - 1; r >= 1; --r)
            if (gm[r] > gm[r + 1]) gm[r] = gm[r + 1];
        auto range_cost = [&](long long s, long long e) {
            if (e <= s) return 0.0;
            const long long r0 = s / U, r1 = (e - 1) / U;
            if (r0 == r1) return gm[(int)(e - s)];
            return gm[(int)(U - s % U)] + (double)(r1 - r0 - 1) * gm[U] + gm[(int)(e - r1 * U)];
        };
        auto cuts_for = [&](double bound, std::vector<long long> *cuts) {
            long long pos = 0;
            for (int q = 0; q < P; ++q) {
                // longest range from pos whose cost stays within the bound
                long long lo = pos, hi = T;
                while (lo < hi) {
                    const long long mid = (lo + hi + 1) / 2;
                    if (range_cost(pos, mid) <= bound + 1e-9) lo = mid; else hi = mid - 1;
                }
                pos = lo;
                if (cuts) cuts->push_back(pos);
                if (pos >= T) break;
            }
            return pos >= T;
        };
        double lo = 0.0, hi = range_cost(0, T);
        for (int it = 0; it < 50; ++it) {
            const double mid = 0.5 * (lo + hi);
            if (cuts_for(mid, nullptr)) hi = mid; else lo = mid;
        }
        std::vector<long long> cuts;
        cuts_for(hi, &cuts);
        // whole tiles round-robin cost 4 per tile: keep them unless the balanced cut is really shorter
        const long long rr_tiles = ((long long)rows * (U / 4) + P - 1) / P;
        if (hi > 0.99 * 4.0 * (double)rr_tiles) cuts.clear();
        long long s = 0;
        for (size_t q = 0; q < cuts.size(); ++q) {
            const long long e = cuts[q];
            while (s < e) {
                const int row = (int)(s / U);
                long long seg_end = (long long)(row + 1) * U;
                if (seg_end > e) seg_end = e;
                int r = (int)(seg_end - s), jj = (int)(s % U);
                while (r > 0) {  // cheapest split of the r units this range owns in this row
                    const int n = first[r];
                    lists[q].push_back(make_int4(row, jj * 64, n * 64, 0));
                    jj += n;
                    r -= n;
                }
                s = seg_end;
            }
        }
    }
    bool any = false;
    for (const auto &l : lists) any = any || !l.empty();
    if (!any) {
        long long t = 0;
        for (int row = 0; row < rows; ++row)
            for (int j = 0; j < U; j += 4, ++t) lists[(size_t)(t % P)].push_back(make_int4(row, j * 64, 256, 0));
    }
    size_t longest = 0;
    for (const auto &l : lists) longest = l.size() > longest ? l.size() : longest;
    stride = (int)longest + 1;
    work.assign((size_t)P * stride, make_int4(0, 0, 0, 0));
    for (int q = 0; q < P; ++q)
        for (size_t i = 0; i < lists[q].size(); ++i) work[(size_t)q * stride + i] = lists[q][i];
}

int pair_plan_init(y2_conv_plan *pl, const y2_conv_desc *d, ConvChoice choice)
{
    if ((d->ksize != 3 && d->ksize != 1) || d->block_k != kPairBK || d->block_n != 256 || d->npad % kPairN ||
        d->cin % kPairBK)
        return Y2_EINVAL;
    const int taps = d->ksize * d->ksize;
    const int hp = d->h + 1, wp = d->w + 1;
    const long long total = (long long)d->batch * hp * wp;
    // wide fp32 heads (yolo9000: 28 269 filters over 1024 channels, a third of that network's step): one-tap form
    // with the staged row-contiguous fp32 stores of conv_epilogue.cuh
    const bool f32_head = taps == 1 && d->out_mode == Y2_OUT_F32_FLAT && d->cout >= 512 && d->out_cs % 4 == 0 &&
                          ((uintptr_t)d->out & 15) == 0;
    // other 1x1 layers: only bf16 tensors through the TMA-store epilogue
    if (taps == 1 && !f32_head && (d->out_mode != Y2_OUT_BF16_PADDED || d->cout % 64)) return Y2_EINVAL;
    // 1x1 layers: the one-tap form of this kernel measured 21.0 us (L19, 1024 -> 512) against 20.1 of the slab kernel,
    // so it is only used when asked for (Y2_CONV_VARIANT=pair; tests).  Keeping the CTA's half of the WHOLE weight
    // matrix in shared memory (yolo-voc L13 / L15, 512 -> 256) halves the L2 -> shared traffic (ncu: 106 -> 68 MB) and
    // still loses, 18.2 us against 16.5 of the slab kernel (profiles/r2o_resident.txt; that resident-weights form was
    // removed later and is in the history) - with three activation stages left the K loop of a 1x1 layer (8 steps of
    // 512 clk per tile) is latency-bound, not traffic-bound.
    if (taps == 1 && choice != kChoosePair && !f32_head) return Y2_EINVAL;
    const int halo = taps == 9 ? wp + 1 : 0;
    const int slab_rows = 128 + 2 * halo;
    const int loads = (slab_rows + 255) / 256;
    int box_rows = (slab_rows + loads - 1) / loads;
    box_rows = (box_rows + 15) / 16 * 16;
    if (box_rows > 256) return Y2_EINVAL;
    const int slab_bytes = loads * box_rows * kPairRowBytes;
    const int aux = ((2 * kPairN * 8 + 512 + 1023) / 1024) * 1024 + 8 * 4096;  // alpha/beta, barriers | store staging
    const int budget = 227 * 1024 - 1024 - aux;
    const int stages_a = taps == 9 ? 2 : kPairMaxStagesA;  // 1x1: a fresh A tile every K step
    int stages_b = (budget - stages_a * slab_bytes) / kPairBHalfBytes;
    if (stages_b > kPairMaxStagesB) stages_b = kPairMaxStagesB;
    if (stages_b < 4) return Y2_EINVAL;
    const int sms = sm_count();
    if (sms < 2) return Y2_EINVAL;
    const int ktot = taps * d->cin;
    int rc = encode_2d_bf16(&pl->tm_a, d->in, (uint64_t)d->cin, (uint64_t)total, (uint64_t)d->in_cs * 2,
                            (uint32_t)kPairBK, (uint32_t)box_rows, kPairBK);
    if (rc == Y2_OK)
        rc = encode_2d_bf16(&pl->tm_b, d->wt, (uint64_t)ktot, (uint64_t)d->npad, (uint64_t)ktot * 2, (uint32_t)kPairBK,
                            128u, kPairBK);
    if (rc != Y2_OK) return rc;
    SlabParams &p = pl->slab;
    p.cblocks = d->cin / kPairBK;
    p.wp = wp;
    p.hp = hp;
    p.h = d->h;
    p.w = d->w;
    p.total_pos = (int)total;
    p.tiles_m = (int)((total + 255) / 256);
    p.tiles_n = d->npad / kPairN;
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
    p.couple = 0;
    p.tma_store = 0;
    memset(&pl->tm_out, 0, sizeof(pl->tm_out));
    if (d->out_mode == Y2_OUT_BF16_PADDED && d->cout % 64 == 0) {
        rc = encode_2d_bf16(&pl->tm_out, d->out, (uint64_t)d->cout, (uint64_t)total, (uint64_t)d->out_cs * 2, 64u, 32u, 64);
        if (rc != Y2_OK) return rc;
        p.tma_store = 1;
    }
    if (f32_head) p.tma_store = 2;
    p.alpha = d->alpha;
    p.beta = d->beta;
    p.out = d->out;
    pl->variant = kVariantPair;
    pl->block_n = kPairN;
    pl->block_k = kPairBK;
    pl->taps = taps;
    pl->smem_bytes = (size_t)stages_a * slab_bytes + (size_t)stages_b * kPairBHalfBytes + aux + 1024;
    const int tiles = p.tiles_m * p.tiles_n;
    const int pairs = tiles < sms / 2 ? tiles : sms / 2;
    pl->grid = 2 * pairs;
    rc = encode_2d_bf16(&pl->tm_b32, d->wt, (uint64_t)ktot, (uint64_t)d->npad, (uint64_t)ktot * 2, (uint32_t)kPairBK,
                        32u, kPairBK);
    if (rc != Y2_OK) return rc;
    std::vector<int4> work;
    int stride = 0;
    const char *bal = getenv("Y2_PAIR_BALANCE");
    pair_schedule(p.tiles_m, d->npad / 64, pairs, !(bal && atoi(bal) == 0), work, stride);
    Y2_CUDA_CHECK(cudaMalloc(&pl->work_buf, work.size() * sizeof(int4)));
    Y2_CUDA_CHECK(cudaMemcpy(pl->work_buf, work.data(), work.size() * sizeof(int4), cudaMemcpyHostToDevice));
    p.work = (const int4 *)pl->work_buf;
    p.work_stride = stride;
    static bool attr_done[64] = {false};
    int dev = 0;
    Y2_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 64 && !attr_done[dev]) {
        Y2_CUDA_CHECK(cudaFuncSetAttribute(conv_pair_kernel<9>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        Y2_CUDA_CHECK(cudaFuncSetAttribute(conv_pair_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        attr_done[dev] = true;
    }
    return Y2_OK;
}

int pair_plan_launch(const y2_conv_plan *pl, cudaStream_t st)
{
    if (pl->taps == 9)
        Y2_CUDA_CHECK(launch_pdl(conv_pair_kernel<9>, dim3(pl->grid), dim3(kPairThreads), pl->smem_bytes, st, pl->tm_a,
                                 pl->tm_b, pl->tm_b32, pl->tm_out, pl->slab));
    else
        Y2_CUDA_CHECK(launch_pdl(conv_pair_kernel<1>, dim3(pl->grid), dim3(kPairThreads), pl->smem_bytes, st, pl->tm_a,
                                 pl->tm_b, pl->tm_b32, pl->tm_out, pl->slab));
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

} // namespace y2

extern "C" int y2_pair_schedule(int rows, int units, int pairs, int balanced, int *out, int cap_entries, int *stride)
{
    if (rows <= 0 || units <= 0 || units % 4 || pairs <= 0 || !out || !stride) return Y2_EINVAL;
    std::vector<int4> work;
    y2::pair_schedule(rows, units, pairs, balanced != 0, work, *stride);
    if ((long long)work.size() > cap_entries) return Y2_EINVAL;
    memcpy(out, work.data(), work.size() * sizeof(int4));
    return (int)work.size();
}
