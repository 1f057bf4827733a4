// Shared device/host helpers for the sm_100a kernels.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "yolo2_b200_kernels.h"

namespace y2 {

void set_error(const char *fmt, ...);

#define Y2_CUDA_CHECK(expr)                                                          \
    do {                                                                             \
        cudaError_t _e = (expr);                                                     \
        if (_e != cudaSuccess) {                                                     \
            y2::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr,               \
                          cudaGetErrorString(_e));                                   \
            return Y2_ECUDA;                                                         \
        }                                                                            \
    } while (0)

#define Y2_LAUNCH_CHECK()                                                            \
    do {                                                                             \
        cudaError_t _e = cudaGetLastError();                                         \
        if (_e != cudaSuccess) {                                                     \
            y2::set_error("%s:%d kernel launch -> %s", __FILE__, __LINE__,           \
                          cudaGetErrorString(_e));                                   \
            return Y2_ECUDA;                                                         \
        }                                                                            \
    } while (0)

static inline cudaStream_t to_stream(y2_stream_t s) { return (cudaStream_t)s; }

int sm_count();

// ---- programmatic dependent launch ---------------------------------------------------
// The layer schedule is a chain of persistent kernels; launched with the programmatic-serialisation attribute, the
// CTAs of layer i+1 are scheduled on an SM as soon as layer i's CTA there has finished: they set up their barriers,
// allocate TMEM and prefetch WEIGHT tiles (which do not depend on layer i) while layer i's last wave drains, and
// only the warp that loads ACTIVATIONS blocks in pdl_wait() until layer i has completed and its stores are visible.
// Without the attribute both instructions are no-ops.
// Only the persistent convolution kernels use it.  Measured (profiles/r2q_pdl_small.txt, A/B in one box): with the
// pool / reorg / shortcut / region / NMS kernels launched the same way the step gets SLOWER (yolo-voc 1.655 -> 1.68 ms,
// resnet50 2.51 -> 2.60, tiny-yolo-voc 0.673 -> 0.698): once all blocks of such a grid have started, the next
// convolution's CTAs (227 KB of shared memory, 59 k registers each) take over the SMs one by one and sit in
// griddepcontrol.wait while the small kernel's tail runs on what is left.
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     Args... args)
{
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// let the next kernel of the stream start its prologue once every CTA of this grid has got this far
__device__ __forceinline__ void pdl_launch_dependents()
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
// block until the kernels this one depends on have completed and their memory operations are visible
__device__ __forceinline__ void pdl_wait()
{
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

// ---- PTX wrappers -----------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count)
                 : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok;
}
// Non-blocking probe (never suspends the thread, unlike try_wait).
__device__ __forceinline__ uint32_t mbar_test_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok;
}
// Bounded wait: a protocol bug becomes a trap (launch failure) instead of a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity, int tag)
{
    if (mbar_try_wait(bar, parity)) return;
    long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) { // ~2 s at 2 GHz
            printf("y2: mbarrier timeout tag=%d block=%d thread=%d parity=%u\n", tag,
                   (int)blockIdx.x, (int)threadIdx.x, parity);
            __trap();
        }
    }
}

// Same, for waiters that are not on the critical path (producers waiting for a free stage, epilogue
// warps waiting for an accumulator): sleep between probes so the spin does not take issue slots
// from the warps that are working on the same SM sub-partition.
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t *bar, uint32_t parity, int tag)
{
    if (mbar_try_wait(bar, parity)) return;
    // watchdog by probe count (every probe sleeps >= 64 ns: 2^25 probes are > 2 s), cheaper in issue slots
    // than reading the clock in kernels whose working warps are issue-bound (first layer, conv+pool)
    unsigned probes = 0;
    while (!mbar_try_wait(bar, parity)) {
        __nanosleep(64);
        if (++probes > (1u << 25)) {
            printf("y2: mbarrier timeout tag=%d block=%d thread=%d parity=%u\n", tag,
                   (int)blockIdx.x, (int)threadIdx.x, parity);
            __trap();
        }
    }
}

// One lane of the (converged) warp gets 1.  Unlike `lane == 0`, ptxas knows a single thread is active
// under this predicate, so the uniform-datapath instructions behind it (UTCHMMA, UTMALDG, UTCBAR)
// are emitted straight-line instead of inside a per-active-thread ELECT/BRA.U.ANY loop.
__device__ __forceinline__ uint32_t elect_one_sync()
{
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .b32 %%rx;\n\t.reg .pred %%px;\n\t"
        "elect.sync %%rx|%%px, %1;\n\t"
        "@%%px mov.s32 %0, 1;\n\t}"
        : "+r"(pred)
        : "r"(0xFFFFFFFFu));
    return pred;
}

__device__ __forceinline__ void fence_barrier_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before()
{
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after()
{
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

__device__ __forceinline__ void tma_prefetch_desc(const void *desc)
{
    asm volatile("prefetch.tensormap [%0];" ::"l"(desc) : "memory");
}

__device__ __forceinline__ void tma_load_2d(const void *desc, uint64_t *bar, void *smem_dst,
                                            int c0, int c1)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
        "l"(desc), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}

// TMA store of one box from shared memory (bulk async-group completion); the issuing thread commits
// the group and later waits until the source buffer may be overwritten
__device__ __forceinline__ void tma_store_2d(const void *desc, const void *smem_src, int c0, int c1)
{
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(desc),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit()
{
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_read()
{
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_all()
{
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// D[tmem] (+)= A[smem] * B[smem], bf16 x bf16 -> fp32, one CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                          uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// All previously issued tcgen05.mma of this thread arrive on `bar` when complete.
__device__ __forceinline__ void umma_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::
                     "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, "
        "[%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
          "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]),
          "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
          "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
          "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]),
          "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait()
{
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---- CTA-pair (cta_group::2) variants -------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// In a cluster launch the shared-window address of a CTA carries its rank in bit 24; clearing it names
// the same offset in the even (leader) CTA of the pair.
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
// TMA load into THIS CTA's shared memory whose completion bytes are credited to the LEADER's mbarrier
__device__ __forceinline__ void tma_load_2d_pair(const void *desc, uint64_t *bar, void *smem_dst, int c0, int c1)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
        "l"(desc), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
        : "memory");
}
// D[tmem of both CTAs] (+)= A[own 128 rows each] * B[N split over both CTAs], issued by the leader only
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// all MMAs issued so far by this thread arrive (once) on the mbarrier at this offset in BOTH CTAs
__device__ __forceinline__ void umma_commit_pair(uint64_t *bar)
{
    const uint16_t mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::
                     "r"(smem_u32(bar)), "h"(mask)
                 : "memory");
}
// arrive on the mbarrier at the same offset in CTA `cta` of the cluster.  Default semantics (release at CTA scope, the
// form cutlass::arch::ClusterBarrier::arrive uses): the explicit .release.cluster costs a MEMBAR.ALL.CTA + ERRBAR per
// arrival (19 % of the samples of a short kernel, profiles/r2p_*), and what the arrival publishes here - "this thread's
// tcgen05.ld of the accumulator has completed" - is ordered by tcgen05.wait::ld + tcgen05.fence::before_thread_sync.
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t *bar, uint32_t cta)
{
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}" ::"r"(smem_u32(bar)),
        "r"(cta)
        : "memory");
}

// K-major shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
// [0,14) start>>4, [16,30) LBO>>4, [32,46) SBO>>4, [46,48) version=1, [61,64) swizzle.
__device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t smem_addr, uint32_t sbo_bytes,
                                                     uint32_t layout_type)
{
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16; // LBO: unused for swizzled K-major, canonical value 1
    d |= (uint64_t)(sbo_bytes >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)layout_type << 61;
    return d;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi)
{
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t *>(&v);
}

} // namespace y2
