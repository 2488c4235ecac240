// Halo-reuse variant of the tcgen05 implicit-GEMM conv3x3 for the high-resolution, narrow layers (Cout = 64 / 128:
// inc.3, down1.*, up3.*, up4.* of reference model/unet.py:72-82). In conv_gemm.cu every tap re-loads its own shifted
// 128-pixel A tile, so a narrow layer moves 9 x 16 KB of activations through L2->SMEM per 128x64 output tile and is
// bound by that fill bandwidth (measured ~450 TFLOP/s). Here one TMA box {64ch, 24, 18, 1} (the 16x16-pixel super
// tile plus its 1-pixel halo, row pitch padded to 24 pixels = 3 swizzle atoms) is loaded ONCE per 64-channel slab and
// all 9 taps x 2 column halves are issued as tcgen05.mma on shifted views of it:
//     A(tap=(dy,dx), half t)  = rows {(h+dy)*24 + (w+dx+8t)},  h in 0..15, w in 0..7   (M = 128 = 16 groups of 8 rows)
//     -> smem descriptor start = stage + (dy*24 + dx + 8t)*128 B, stride-byte-offset = 24*128 = 3072 B.
// The start address is no longer 1024 B aligned when dx != 0; the 128B-swizzle XOR is a function of the absolute smem
// address bits [7,10), which is also what TMA used when it wrote the box, so the shifted view reads the right chunks
// (validated on B200 against the oracle; putting the row phase into the descriptor's base-offset field instead is wrong).
// Weights stream per (tap, slab) through their own ring. Warp roles (224 threads, 352 with two epilogue sets): 0 = A
// producer, 1 = TMEM owner + MMA issuer, 2 = B producer, 3.. = epilogue. TMEM: 2 accumulator sets x 2 halves x Cout
// columns.
//
// CTA pairs (conv_halo2_kernel, cta_group::2). The narrow layers are bound by shared-memory bandwidth: a single-CTA
// tcgen05.mma of N = 64 reads 4 KB of A and 2 KB of B per 32 tensor-pipe cycles (measured 50.8 cycles per instruction,
// tools/probe/mma_probe.cu), N = 128 reads 8 KB per 64 cycles while TMA fills compete for the same port. In a CTA pair
// each SM keeps its own super tile's halo (A) but only HALF of every weight slab (Cout/2 rows); the M256 x Cout
// instruction reads both halves. That halves the weight traffic per SM (fills and operand reads), and it lets the
// weights of two more layers stay resident (up4.conv.0: 144 KB -> 72 KB per SM; down1.conv.0: 144 KB -> 72 KB).
// Protocol: as the per-tap pair in conv_gemm.cu. Both CTAs run the same code on adjacent super tiles (rank picks the
// tile); producers wait on local "empty" barriers and send completion bytes to the leader's "full" barriers; the leader
// issues every MMA and commits with a multicast to both CTAs; epilogue warps of both CTAs release the accumulator on
// the leader.
#include "conv_epilogue.cuh"
#include "conv_gemm.cuh"
#include "ptx.cuh"

#include <cstdio>
#include <cstring>

namespace fi {

namespace {

constexpr int HT = 16;                                 // super tile: 16 x 16 output pixels
constexpr int HALO_W = 24, HALO_H = 18;                // TMA box (pixels): 16+2 columns padded to 24, 16+2 rows
constexpr int HALO_BYTES = HALO_W * HALO_H * 128;      // 55296
constexpr int HALO_THREADS = 224;        // 3 role warps + 4 epilogue warps (precise mode)
constexpr int HALO_THREADS_8 = 352;      // 3 role warps + 8 epilogue warps (one set per column half)
constexpr int A_STAGES = 2;
constexpr int PREFETCH_DIST = 2;         // L2-prefetch the halo boxes this many grid strides ahead (DESIGN §3 item 3)
constexpr int B_RING_BYTES = 65536;      // streamed weights: a ring of weight slices
constexpr int B_REGION_BYTES = 73728;    // weight region: the ring, or up to 72 KB of resident weight slices
constexpr int H_STAGING_PER_WARP = 2 * 4096;
constexpr int H_POOL_PER_WARP = 2 * 1024;
constexpr int H_BAR_BYTES = 512;
constexpr int HALO_SMEM =
    1024 + A_STAGES * HALO_BYTES + B_REGION_BYTES + 4 * (H_STAGING_PER_WARP + H_POOL_PER_WARP) + H_BAR_BYTES;
static_assert(HALO_SMEM <= 232448, "halo kernel exceeds the 227 KB shared memory limit");

// One weight slice: this CTA's rows (all Cout, or half of them in a CTA pair) of one [Cout x 64] (tap, slab) slab.
__host__ __device__ constexpr int halo_b_stage_bytes(int ctas, int cout) { return cout / ctas * 128; }
// RESIDENT: all 9 x slabs weight slices this CTA holds fit in the weight region and stay for the CTA's lifetime.
__host__ __device__ constexpr bool halo_resident_fits(int ctas, int cout, int slabs) {
    return 9 * slabs * halo_b_stage_bytes(ctas, cout) <= B_REGION_BYTES;
}

__device__ __forceinline__ uint64_t halo_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
    d |= static_cast<uint64_t>(1) << 16;
    d |= static_cast<uint64_t>((HALO_W * 128) >> 4) << 32;  // 3072 B between consecutive tile rows (8-row groups)
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}

struct Unit {
    HaloTile t;
    bool valid;  // false: odd tile count, the last pair's second CTA recomputes the last tile with its stores off
};
template <int CTAS>
__device__ __forceinline__ Unit decode_unit(int u, uint32_t rank, const ConvKernelParams& p) {
    const int per_img = p.tiles_y * p.tiles_x;
    const int tiles = p.n_img * per_img;
    int m = CTAS * u + static_cast<int>(rank);
    Unit r;
    r.valid = CTAS == 1 || m < tiles;
    if (!r.valid) m = tiles - 1;
    r.t.img = m / per_img;
    m -= r.t.img * per_img;
    const int ty = m / p.tiles_x;
    r.t.y0 = ty * HT;
    r.t.x0 = (m - ty * p.tiles_x) * HT;
    return r;
}

// CTAS = 1: one CTA per super tile. CTAS = 2: a CTA pair (cluster of 2) computes two adjacent super tiles.
template <int CTAS, int COUT, int MODE, bool RESIDENT, bool SPLIT>
__device__ __forceinline__ void conv_halo_body(const ConvMaps& maps, const ConvKernelParams& p) {
    constexpr int B_STAGE_BYTES = halo_b_stage_bytes(CTAS, COUT);
    constexpr int B_STAGES = B_RING_BYTES / B_STAGE_BYTES;  // ring depth when streaming
    constexpr int ACC_COLS = 2 * COUT;          // two column halves
    constexpr int TMEM_COLS = 2 * ACC_COLS;     // double buffered: 256 (Cout 64) or 512 (Cout 128)
    constexpr uint32_t IDESC = umma_idesc_bf16(128 * CTAS, COUT);
    static_assert(MODE != EPI_HEAD || COUT == 64, "head epilogue consumes exactly 64 channels");
    // bf16 mode: 8 epilogue warps, one set of 4 per column half, single staging tile each; precise mode: 4 warps
    constexpr int EPI_SETS = SPLIT ? 1 : 2;
    constexpr int STAGE_PER_WARP = SPLIT ? 2 * 4096 : 4096;
    constexpr int POOL_PER_WARP = SPLIT ? 2 * 1024 : 1024;

    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t smem_a = smem_base;
    const uint32_t smem_b = smem_a + A_STAGES * HALO_BYTES;
    const uint32_t smem_stage = smem_b + B_REGION_BYTES;
    const uint32_t smem_pool = smem_stage + 4 * H_STAGING_PER_WARP;
    const uint32_t smem_bar = smem_pool + 4 * H_POOL_PER_WARP;
    const uint32_t bar_afull = smem_bar;                       // A_STAGES
    const uint32_t bar_aempty = bar_afull + 8 * A_STAGES;      // A_STAGES
    const uint32_t bar_bfull = bar_aempty + 8 * A_STAGES;      // B_STAGES
    const uint32_t bar_bempty = bar_bfull + 8 * B_STAGES;      // B_STAGES
    const uint32_t bar_tfull = bar_bempty + 8 * B_STAGES;      // 2
    const uint32_t bar_tempty = bar_tfull + 16;                // 2
    const uint32_t bar_bres = bar_tempty + 16;                 // 1 (RESIDENT: all weights landed)
    const uint32_t tmem_slot = bar_bres + 8;
    uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = CTAS == 1 ? 0 : cluster_ctarank();
    const bool leader = CTAS == 1 || rank == 0;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&maps.a[0]);
        tma_prefetch_desc(&maps.a[2]);
        tma_prefetch_desc(&maps.b);
        if (MODE != EPI_HEAD) tma_prefetch_desc(&maps.out[0]);
        if (MODE == EPI_STORE_POOL) tma_prefetch_desc(&maps.pool[0]);
        for (int s = 0; s < A_STAGES; ++s) {
            mbar_init(bar_afull + 8 * s, 1);
            mbar_init(bar_aempty + 8 * s, 1);
        }
        for (int s = 0; s < B_STAGES; ++s) {
            mbar_init(bar_bfull + 8 * s, 1);
            mbar_init(bar_bempty + 8 * s, 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(bar_tfull + 8 * a, 1);
            mbar_init(bar_tempty + 8 * a, 4 * EPI_SETS * CTAS);  // one arrive per epilogue warp (of both CTAs)
        }
        mbar_init(bar_bres, 1);
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc<CTAS>(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    if constexpr (CTAS == 2) cluster_sync_all();  // both CTAs' barriers exist before any remote signal can arrive
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    pdl_launch_dependents();
    pdl_wait();

    const int units = (p.n_img * p.tiles_y * p.tiles_x + CTAS - 1) / CTAS;
    const int unit0 = static_cast<int>(blockIdx.x / CTAS);
    const int unit_step = static_cast<int>(gridDim.x / CTAS);
    const int slabs = p.slabs;
    const int b_row0 = static_cast<int>(rank) * (COUT / CTAS);  // this CTA's rows of every weight slab

    if (warp == 0) {
        // ------------------------------------------------------------ A producer: one halo box per (tile, slab)
        {
            int stage = 0;
            uint32_t phase = 0;
            for (int u = unit0; u < units; u += unit_step) {
                const HaloTile tc = decode_unit<CTAS>(u, rank, p).t;
                // Only A_STAGES-1 halo boxes can be in flight towards smem, which does not cover HBM latency:
                // pull the boxes of this CTA's tile after next into L2 now (no smem needed for that).
                const int up = u + PREFETCH_DIST * unit_step;
                if (up < units && lane == 0) {
                    const HaloTile pc = decode_unit<CTAS>(up, rank, p).t;
                    for (int g = 0; g < p.nseg; ++g) {
                        const int mid = p.seg_map[g];
                        if (g > 0 && p.seg_map[g - 1] == mid) continue;  // same tensor as the previous segment
                        const int ox = mid >= 2 ? p.off_x : 0, oy = mid >= 2 ? p.off_y : 0;
                        for (int c = 0; c < p.seg_slabs[g]; ++c)
                            tma_prefetch_l2_4d(&maps.a[mid], c * BLOCK_K, pc.x0 - 1 - ox, pc.y0 - 1 - oy, pc.img);
                    }
                }
                int seg = 0, left = p.seg_slabs[0];
                for (int s = 0; s < slabs; ++s) {
                    while (left == 0) left = p.seg_slabs[++seg];
                    const int local = p.seg_slabs[seg] - left;
                    --left;
                    const int mid = p.seg_map[seg];
                    mbar_wait(bar_aempty + 8 * stage, phase ^ 1);
                    const uint32_t full = bar_afull + 8 * stage;
                    if (elect_one()) {
                        if (leader) mbar_expect_tx(full, CTAS * HALO_BYTES);
                        const int ox = mid >= 2 ? p.off_x : 0, oy = mid >= 2 ? p.off_y : 0;  // F.pad of src1
                        tma_load_4d<CTAS>(smem_a + stage * HALO_BYTES, &maps.a[mid], full, local * BLOCK_K,
                                          tc.x0 - 1 - ox, tc.y0 - 1 - oy, tc.img);
                    }
                    __syncwarp();
                    if (++stage == A_STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 2) {
        // ------------------------------------------------------------ B producer: one weight slice per (slab, tap)
        if (RESIDENT) {
            if (lane == 0) {
                const int res_slabs = CTAS == 1 ? 1 : slabs;  // a single CTA holds Cout 64 x Cin 64 only (72 KB)
                if (leader) mbar_expect_tx(bar_bres, CTAS * 9 * res_slabs * B_STAGE_BYTES);
                for (int s = 0; s < res_slabs; ++s)
                    for (int tap = 0; tap < 9; ++tap)
                        tma_load_2d<CTAS>(smem_b + (s * 9 + tap) * B_STAGE_BYTES, &maps.b, bar_bres,
                                          (tap * slabs + s) * BLOCK_K, b_row0);
            }
        } else {
            int stage = 0;
            uint32_t phase = 0;
            for (int u = unit0; u < units; u += unit_step) {
                for (int s = 0; s < slabs; ++s) {
                    for (int tap = 0; tap < 9; ++tap) {
                        mbar_wait(bar_bempty + 8 * stage, phase ^ 1);
                        const uint32_t full = bar_bfull + 8 * stage;
                        if (elect_one()) {
                            if (leader) mbar_expect_tx(full, CTAS * B_STAGE_BYTES);
                            tma_load_2d<CTAS>(smem_b + stage * B_STAGE_BYTES, &maps.b, full,
                                              (tap * slabs + s) * BLOCK_K, b_row0);
                        }
                        __syncwarp();
                        if (++stage == B_STAGES) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer (warp converged, one elected lane
        // issues; a pair's MMAs are all issued by the leader CTA)
        if (leader) {
            int a_stage = 0, b_stage = 0;
            uint32_t a_phase = 0, b_phase = 0;
            int it = 0;
            if (RESIDENT) mbar_wait(bar_bres, 0);
            for (int u = unit0; u < units; u += unit_step, ++it) {
                const int acc = it & 1;
                const uint32_t acc_phase = (it >> 1) & 1;
                mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * ACC_COLS;
                for (int s = 0; s < slabs; ++s) {
                    mbar_wait(bar_afull + 8 * a_stage, a_phase);
                    const uint32_t a_base = smem_a + a_stage * HALO_BYTES;
                    for (int tap = 0; tap < 9; ++tap) {
                        if (!RESIDENT) mbar_wait(bar_bfull + 8 * b_stage, b_phase);
                        tc_fence_after();
                        const int dy = tap / 3, dx = tap - 3 * dy;
                        const uint64_t db =
                            umma_desc_sw128(smem_b + (RESIDENT ? s * 9 + tap : b_stage) * B_STAGE_BYTES);
                        const uint64_t da0 = halo_desc(a_base + (dy * HALO_W + dx) * 128);
                        if (elect_one()) {
                            // The two column halves are independent accumulators: alternating them keeps back-to-back
                            // tcgen05.mma from serialising on the same TMEM tile.
#pragma unroll
                            for (int k = 0; k < BLOCK_K / 16; ++k) {
#pragma unroll
                                for (int half = 0; half < 2; ++half) {
                                    // +8 pixels (1024 B) per column half, +32 B per K step, in 16-byte units
                                    umma_bf16_ss<CTAS>(d_tmem + half * COUT, da0 + 64 * half + 2 * k, db + 2 * k,
                                                       IDESC, (s | tap | k) != 0);
                                }
                            }
                            if (!RESIDENT) umma_commit<CTAS>(bar_bempty + 8 * b_stage);
                            if (tap == 8) {
                                umma_commit<CTAS>(bar_aempty + 8 * a_stage);
                                if (s == slabs - 1) umma_commit<CTAS>(bar_tfull + 8 * acc);
                            }
                        }
                        __syncwarp();
                        if (!RESIDENT) {
                            if (++b_stage == B_STAGES) {
                                b_stage = 0;
                                b_phase ^= 1;
                            }
                        }
                    }
                    if (++a_stage == A_STAGES) {
                        a_stage = 0;
                        a_phase ^= 1;
                    }
                }
            }
        }
    } else {
        // ------------------------------------------------------------ epilogue warps 3..6 (3..10 with two sets)
        const int q = warp & 3;  // TMEM lanes [32q, 32q+32) <-> tile rows 4q..4q+3, 8 columns of one half
        const int ew = warp - 3;          // 0..7 (0..3 in precise mode)
        const int set = ew >> 2;          // which column half this warp drains (bf16 mode)
        const uint32_t my_stage = smem_stage + ew * STAGE_PER_WARP;
        const uint32_t my_pool = smem_pool + ew * POOL_PER_WARP;
        int buf = 0;
        int it = 0;
        for (int u = unit0; u < units; u += unit_step, ++it) {
            const Unit w = decode_unit<CTAS>(u, rank, p);
            const int acc = it & 1;
            const uint32_t acc_phase = (it >> 1) & 1;
            mbar_wait(bar_tfull + 8 * acc, acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * ACC_COLS;
#pragma unroll 1
            for (int c = set * (ACC_COLS / 64 / EPI_SETS); c < (set + 1) * (ACC_COLS / 64 / EPI_SETS); ++c) {
                epilogue_chunk_halo<COUT, MODE, SPLIT, SPLIT>(maps, p, w.t, taddr, c, q, lane, my_stage, my_pool, buf,
                                                              w.valid);
            }
            tc_fence_before();
            __syncwarp();
            if (elect_one()) {
                if (leader) mbar_arrive(bar_tempty + 8 * acc);
                else mbar_arrive_cluster(bar_tempty + 8 * acc, 0);
            }
        }
        __syncwarp();
        if (MODE != EPI_HEAD && elect_one()) tma_store_wait_all();
    }

    tc_fence_before();
    __syncthreads();
    if constexpr (CTAS == 2) cluster_sync_all();  // the peer may still be reading TMEM / receiving commits
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<CTAS>(tmem_base, TMEM_COLS);
    }
}

template <int COUT, int MODE, bool RESIDENT, bool SPLIT>
__global__ void __launch_bounds__(SPLIT ? HALO_THREADS : HALO_THREADS_8, 1)
conv_halo_kernel(const __grid_constant__ ConvMaps maps, const ConvKernelParams p) {
    conv_halo_body<1, COUT, MODE, RESIDENT, SPLIT>(maps, p);
}

template <int COUT, int MODE, bool RESIDENT, bool SPLIT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(SPLIT ? HALO_THREADS : HALO_THREADS_8, 1)
conv_halo2_kernel(const __grid_constant__ ConvMaps maps, const ConvKernelParams p) {
    conv_halo_body<2, COUT, MODE, RESIDENT, SPLIT>(maps, p);
}

template <int CTAS, int COUT, int MODE, bool RESIDENT = false, bool SPLIT = false>
const char* launch_inst(const ConvLaunch& l, cudaStream_t stream) {
    if constexpr (!SPLIT && !RESIDENT && MODE != EPI_HEAD) {
        if (l.split) return launch_inst<CTAS, COUT, MODE, false, true>(l, stream);
    }
    // Only where some layer can satisfy the rule: a precise-mode layer has at least 3 slabs.
    if constexpr (!RESIDENT && halo_resident_fits(CTAS, COUT, SPLIT ? 3 : 1)) {
        if (halo_resident_fits(CTAS, COUT, l.p.slabs)) return launch_inst<CTAS, COUT, MODE, true, SPLIT>(l, stream);
    }
    void (*kfn)(ConvMaps, ConvKernelParams);
    if constexpr (CTAS == 1) kfn = conv_halo_kernel<COUT, MODE, RESIDENT, SPLIT>;
    else kfn = conv_halo2_kernel<COUT, MODE, RESIDENT, SPLIT>;
    static std::atomic<uint64_t> configured{0};  // per instantiation: devices with the shared-memory opt-in
    if (!smem_opt_in(kfn, HALO_SMEM, configured)) return "cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed";
    const cudaError_t e = launch_kernel(kfn, dim3(l.grid), dim3(SPLIT ? HALO_THREADS : HALO_THREADS_8), HALO_SMEM,
                                        stream, l.maps, l.p);
    return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

template <int CTAS>
const char* launch_halo(const ConvLaunch& l, cudaStream_t stream) {
    switch (l.block_n * 4 + l.mode) {
        case 64 * 4 + EPI_STORE: return launch_inst<CTAS, 64, EPI_STORE>(l, stream);
        case 64 * 4 + EPI_STORE_POOL: return launch_inst<CTAS, 64, EPI_STORE_POOL>(l, stream);
        case 64 * 4 + EPI_HEAD: return launch_inst<CTAS, 64, EPI_HEAD>(l, stream);
        case 128 * 4 + EPI_STORE: return launch_inst<CTAS, 128, EPI_STORE>(l, stream);
        case 128 * 4 + EPI_STORE_POOL: return launch_inst<CTAS, 128, EPI_STORE_POOL>(l, stream);
        default: return "conv(halo): no kernel instantiation for this (cout, mode)";
    }
}

}  // namespace

bool conv_halo_eligible(const ConvDesc& d) {
    if (d.taps != 9) return false;
    if (d.n_total != 64 && d.n_total != 128) return false;
    if (d.mode == EPI_HEAD) return d.n_total == 64;
    return d.mode == EPI_STORE || d.mode == EPI_STORE_POOL;
}

void conv_halo_geometry(int* tile, int* box_w, int* box_h, int* out_w, int* out_h, int* pool_w, int* pool_h) {
    *tile = HT;
    *box_w = HALO_W;
    *box_h = HALO_H;
    *out_w = 8;
    *out_h = 4;
    *pool_w = 4;
    *pool_h = 2;
}

const char* conv_halo_launch(const ConvLaunch& l, cudaStream_t stream) {
    return l.pair ? launch_halo<2>(l, stream) : launch_halo<1>(l, stream);
}

}  // namespace fi
