// Thin inline-PTX wrappers for the sm_100a features the frame-synthesis kernels use:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM alloc / TMEM load / commit).
// Everything here is device-only and header-only.
#pragma once
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <utility>
#include <cuda.h>
#include <cuda_runtime.h>

namespace fi {

// Host helper: cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute of a kernel, and one process may
// drive several GPUs (one fiNet + one worker thread per device). `done` is the per-instantiation bit mask of devices
// that already have the opt-in; safe to call from several threads.
// FI_PDL=0 turns programmatic dependent launch off (plain stream order), e.g. to A/B its effect.
inline bool pdl_enabled() {
    const char* e = getenv("FI_PDL");  // read per launch (tens of ns) so that tests can flip it
    return e ? e[0] != '0' : true;
}

// Launch of a kernel that calls pdl_wait() before its first dependent memory access.
template <class... KArgs, class... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                 Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

template <class Kernel>
inline bool smem_opt_in(Kernel kfn, int bytes, std::atomic<uint64_t>& done) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return false;
    const uint64_t bit = 1ull << (dev & 63);
    if (done.load(std::memory_order_acquire) & bit) return true;
    if (cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) != cudaSuccess) return false;
    done.fetch_or(bit, std::memory_order_release);
    return true;
}

#ifndef FI_WAIT_WATCHDOG
#define FI_WAIT_WATCHDOG (1u << 26)   // bounded spins before a role gives up and traps (no silent hangs)
#endif

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// One lane of a fully converged warp (elect.sync): lets the compiler keep descriptors in uniform registers and emit
// straight-line UTCHMMA / UTMALDG sequences instead of per-instruction election loops.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

// ------------------------------------------------------------------ programmatic dependent launch (PDL)
// Kernels of the forward schedule are launched with cudaLaunchAttributeProgrammaticStreamSerialization (launch_kernel
// below): the next layer's CTAs may be scheduled onto SMs that the current layer has already vacated and run their
// prologue (barrier init, TMEM allocation, descriptor prefetch) there. pdl_wait() blocks until the preceding grid has
// COMPLETED and its memory is visible, so everything after it is ordered exactly as without PDL; nothing before it may
// touch memory another kernel produces or consumes. pdl_launch_dependents() lets the grid after this one start its
// own prologue early. Both are no-ops when the kernel was launched without the attribute.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug turns into a trap (sticky launch error) instead of a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > FI_WAIT_WATCHDOG) {
            printf("fi_b200: mbarrier watchdog block %d thread %d bar 0x%x parity %u\n", (int)blockIdx.x,
                   (int)threadIdx.x, bar, parity);
            __trap();
        }
    }
}

// ------------------------------------------------------------------ proxies / fences
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ------------------------------------------------------------------ CTA pairs (cta_group::2, cluster of 2)
// A shared::cta address carries the CTA's rank within the pair in bit 24 when used as a shared::cluster address;
// clearing it addresses the same offset in CTA 0 (the MMA leader).
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {  // every thread of both CTAs
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// Arrive on the mbarrier at the same offset in CTA `cta` of the cluster.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t cta) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}"
        ::"r"(bar), "r"(cta)
        : "memory");
}

// ------------------------------------------------------------------ TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// CTAS = 1: data and completion bytes go to this CTA. CTAS = 2 (CTA pair): data lands in the executing CTA's smem,
// completion bytes go to the LEADER's mbarrier.
template <int CTAS = 1>
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
    if constexpr (CTAS == 1) {
        asm volatile(
            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
            ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
            : "memory");
    } else {
        asm volatile(
            "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
            "%4}], [%2];" ::"r"(dst),
            "l"(reinterpret_cast<uint64_t>(m)), "r"(bar & PEER_BIT_MASK), "r"(c0), "r"(c1)
            : "memory");
    }
}
template <int CTAS = 1>
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
    if constexpr (CTAS == 1) {
        asm volatile(
            "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
            "[%2];" ::"r"(dst),
            "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
            : "memory");
    } else {
        asm volatile(
            "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
            "%4, %5, %6}], [%2];" ::"r"(dst),
            "l"(reinterpret_cast<uint64_t>(m)), "r"(bar & PEER_BIT_MASK), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
            : "memory");
    }
}
// Pull a box into L2 only (no smem, no barrier): lets the real load of a later tile hit L2 instead of HBM.
__device__ __forceinline__ void tma_prefetch_l2_4d(const CUtensorMap* m, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.prefetch.tensor.4d.L2.global.tile [%0, {%1, %2, %3, %4}];" ::"l"(
                     reinterpret_cast<uint64_t>(m)),
                 "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(m)),
                 "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2, int c3,
                                             int c4) {
    asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(m)),
                 "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ------------------------------------------------------------------ TMEM
// One full warp executes alloc / dealloc (.sync.aligned); in a CTA pair (CTAS = 2) the same warp of both CTAs.
template <int CTAS = 1>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
    if constexpr (CTAS == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    } else {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
}
template <int CTAS = 1>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    if constexpr (CTAS == 1)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
    else
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive fp32 columns: thread t of the warp receives lane (base_lane + t).
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}

// ------------------------------------------------------------------ tcgen05.mma (bf16/f16 -> fp32)
// D[tmem] (+)= A[smem desc] * B[smem desc]; issued by ONE thread. CTAS = 2: D[256 x N] (+)= A[256 x 16] * B[N x 16]^T
// over the CTA pair, each CTA holding its own 128 rows of A and half of B; issued by one thread of the leader CTA.
template <int CTAS = 1>
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
    if constexpr (CTAS == 1) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
            : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
            : "memory");
    }
}
// Arrive on an mbarrier once every previously issued tcgen05.mma of this thread has completed
// (implies tcgen05.fence::before_thread_sync). CTAS = 2: on the mbarrier at this offset in BOTH CTAs.
template <int CTAS = 1>
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    if constexpr (CTAS == 1) {
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
                     : "memory");
    } else {
        asm volatile(
            "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
            ::"r"(bar), "h"(static_cast<uint16_t>(3))
            : "memory");
    }
}

// K-major, 128-byte-swizzled operand tile (rows of 128 B, 8-row atoms of 1024 B):
//   bits [0,14)  start address >> 4        bits [16,30) leading byte offset >> 4 (ignored for swizzled K-major; 1)
//   bits [32,46) stride byte offset >> 4   (1024 B between 8-row groups)
//   bits [46,48) descriptor version = 1 (Blackwell)   bits [61,64) layout type 2 = SWIZZLE_128B
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
    d |= static_cast<uint64_t>(1) << 16;
    d |= static_cast<uint64_t>(1024 >> 4) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}
// Instruction descriptor, kind::f16: fp32 accumulate, bf16 A/B, both K-major, dense.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(N >> 3) << 17) |
           (static_cast<uint32_t>(M >> 4) << 24);
}

// ------------------------------------------------------------------ small helpers
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t bf16x2_max(uint32_t a, uint32_t b) {
    uint32_t r;
    asm("max.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
    return r;
}

// ------------------------------------------------------------------ precise mode helpers (value = bf16 hi + bf16 lo)
__device__ __forceinline__ float bf16lo_f(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16hi_f(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }

// 64 fp32 values -> 32 packed bf16x2 hi words + 32 packed lo words (lo = bf16(f - hi): ~16 mantissa bits in total)
__device__ __forceinline__ void split_hi_lo(const float (&f)[64], uint32_t (&hi)[32], uint32_t (&lo)[32]) {
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        const uint32_t h = pack_bf16x2(f[2 * j], f[2 * j + 1]);
        hi[j] = h;
        lo[j] = pack_bf16x2(f[2 * j] - bf16lo_f(h), f[2 * j + 1] - bf16hi_f(h));
    }
}

// 2x2 max-pool of (hi, lo) pairs: 16-byte chunk j of four staged rows (128B-swizzled staging tiles shi / slo).
// hi + lo is exact in fp32 (<= 17 significant bits), so the max is taken on the true values and re-split.
__device__ __forceinline__ void pool4_hi_lo(uint32_t shi, uint32_t slo, const int (&rows)[4], int j, uint4& mh,
                                            uint4& ml) {
    float m[8];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const uint32_t off = rows[r] * 128 + ((j ^ (rows[r] & 7)) << 4);
        const uint4 h = ld_shared_v4(shi + off);
        const uint4 l = ld_shared_v4(slo + off);
        const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const float v0 = bf16lo_f(hw[w]) + bf16lo_f(lw[w]);
            const float v1 = bf16hi_f(hw[w]) + bf16hi_f(lw[w]);
            m[2 * w] = r == 0 ? v0 : fmaxf(m[2 * w], v0);
            m[2 * w + 1] = r == 0 ? v1 : fmaxf(m[2 * w + 1], v1);
        }
    }
    uint32_t oh[4], ol[4];
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        oh[w] = pack_bf16x2(m[2 * w], m[2 * w + 1]);
        ol[w] = pack_bf16x2(m[2 * w] - bf16lo_f(oh[w]), m[2 * w + 1] - bf16hi_f(oh[w]));
    }
    mh = make_uint4(oh[0], oh[1], oh[2], oh[3]);
    ml = make_uint4(ol[0], ol[1], ol[2], ol[3]);
}

}  // namespace fi
